"""Parity pin against REFERENCE-HELD code: the reference's own CUDA kernels (sp1-gpu/crates/sys/lib/**, compiled unmodified into
oracle/_ref/libsp1ref.so by oracle/Makefile, launched with the reference's grid/block shapes by oracle/ref_launcher.cu) were run on
the seeded inputs below; what they returned is stored in tests/golden/ref_kernels.json (SHA-256 of every output array, the words
themselves where a test needs the values) by tools/gen_ref_kernels_golden.py.  Each test compares (a) the CPU oracle and (b) the
product library through its C ABI with those stored outputs.  Everything is bit-exact.
Covers SURVEY.md §8 rows T1 (field, Poseidon2, sponge, compress, DuplexChallenger, grind), A3 (batch_coset_dft), A4 (leafHashPacked +
compress tree), the BaseFold / multilinear primitives of A5 (batchKernel, foldMle, fixLastVariable, partial_lagrange), the LogUp-GKR
first-layer interaction evaluation of A8 (populateLastCircuitLayer) and the zerocheck constraint-bytecode interpreter of A7
(zerocheck_fused_sequential)."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

from tests import oracle_lib as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_kernels.json")
pytestmark = pytest.mark.gpu

WORDS_UP_TO = 64   # outputs this small are stored word for word, larger ones as SHA-256 + shape

MERKLE_SHAPES = [(1, 1), (3, 4), (8, 6), (9, 7), (16, 9), (91, 10), (24, 13), (95, 12), (192, 8)]
DFT_SHAPES = [(2, 1, 2), (3, 3, 1), (5, 4, 2), (8, 2, 2), (10, 3, 2), (11, 2, 2), (12, 3, 2), (13, 1, 3), (14, 2, 2), (16, 2, 2), (18, 2, 2),
              (19, 1, 2), (20, 1, 2), (21, 2, 2)]
SPONGE_WIDTHS = [1, 2, 7, 8, 9, 15, 16, 17, 24, 91]
GRIND_BITS = [1, 5, 12, 16, 20]
LAGRANGE_VARS = [1, 2, 5, 11]
GKR_CHIPS = [("tinyc", "Add", 64), ("tinyc", "Byte", 96), ("tinyc", "DivRem", 32), ("tinyr", "ExtAlu", 128)]
ZEROCHECK_CHIPS = [("tinyc", "Add", 64), ("tinyc", "Byte", 2048), ("tinyc", "Mul", 4096), ("tinyr", "Poseidon2Wide", 512)]


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype="<u4").tobytes()).hexdigest()


def golden_entry(a):
    """what the golden file keeps of one reference output"""
    a = np.ascontiguousarray(a, np.uint32)
    e = {"shape": list(a.shape), "sha256": digest(a)}
    if a.size <= WORDS_UP_TO:
        e["words"] = [int(x) for x in a.reshape(-1)]
    return e


_gold = None


def _ref(key):
    global _gold
    if _gold is None:
        _gold = json.load(open(GOLDEN))["outputs"]
    return _gold[key]


def ref_words(key):
    e = _ref(key)
    return np.array(e["words"], np.uint32).reshape(e["shape"])


def same_as_ref(key, a):
    e = _ref(key)
    return list(np.shape(a)) == e["shape"] and digest(a) == e["sha256"]


# ---- the seeded inputs the reference kernels were run on ---------------------------------------------------------------------------------
def _edge_field(rng, n):
    a = O.rand_field(rng, n)
    a[:6] = [0, 1, O.P - 1, 0x01FFFFFE, 0x7F000000, 2]   # 0, tiny, p-1 (raw words), ONE, p-1, 2
    return a


def field_inputs():
    rng = np.random.default_rng(1)
    n = 4096
    return _edge_field(rng, n), _edge_field(rng, n)[::-1].copy()


def ext_inputs():
    rng = np.random.default_rng(2)
    n = 2048
    a, b = O.rand_field(rng, (n, 4)), O.rand_field(rng, (n, 4))
    a[0] = 0; a[1] = [0x01FFFFFE, 0, 0, 0]; b[2] = 0; a[3] = O.to_monty(np.full(4, O.P - 1))
    return a, b, O.rand_field(rng, (n, 4))


def permute_inputs():
    rng = np.random.default_rng(3)
    st = O.rand_field(rng, (3000, 16))
    st[0] = 0
    st[1] = O.to_monty(np.full(16, O.P - 1))
    st[2] = 0x01FFFFFE
    return st


def sponge_inputs(n_in):
    return O.rand_field(np.random.default_rng(10 + n_in), (64, n_in))


def merkle_inputs(width, log_h):
    return O.rand_field(np.random.default_rng(200 + width), (width, 1 << log_h))


def dft_inputs(log_h, ncols):
    return O.rand_field(np.random.default_rng(300 + log_h), (ncols, 1 << log_h))


def dft_max_inputs():
    return O.rand_field(np.random.default_rng(321), (1, 1 << 21))


def challenger_inputs():
    rng = np.random.default_rng(5)
    n = 400
    ops = rng.choice([0, 0, 0, 1, 1, 2], size=n).astype(np.uint32)
    vals = O.rand_field(rng, n)
    vals[ops == 2] = rng.integers(1, 24, size=int((ops == 2).sum()))
    return ops, vals


def grind_inputs(bits):
    rng = np.random.default_rng(600 + bits)
    ch = O.Challenger()
    ch.observe(O.rand_field(rng, 11))
    ch.sample(3)
    ch.observe(O.rand_field(rng, 2))
    return ch


def batch_inputs():
    rng = np.random.default_rng(7)
    width, height = 13, 1 << 9
    return O.rand_field(rng, (width, height)), O.rand_field(rng, (width, 4))


def fold_inputs():
    rng = np.random.default_rng(8)
    m = 1 << 10
    return O.rand_field(rng, (2 * m, 4)), O.rand_field(rng, 4)


def lagrange_inputs(n_vars):
    return O.rand_field(np.random.default_rng(9 + n_vars), (n_vars, 4))


def _chip(workload, chip_name, h, seed):
    from sp1_b200 import synth_air as SA
    from sp1_b200 import workload as W
    m = W.synthetic_machine(workload, seed=42)
    k = m["names"].index(chip_name)
    sp = m["specs"][k]
    rng = np.random.default_rng(seed)
    main, prep = SA.synth_trace(rng, h, sp.g, sp.wp, 12345, extra_cols=sp.extra, extra_prep=sp.extra_prep)
    return m, k, main, prep, rng


def gkr_inputs(workload, chip_name, h):
    m, k, main, prep, rng = _chip(workload, chip_name, h, 77 + h)
    alpha = O.rand_field(rng, 4)
    betas = O.rand_field(rng, (16, 4))
    return m, k, main, prep, alpha, betas


def zerocheck_inputs(workload, chip_name, h):
    from tests import ref_lib as R   # blob parsing only (plain Python, no reference library)
    m, k, main, prep, rng = _chip(workload, chip_name, h, 99 + h)
    chip = R.parse_chip_words(m["blob"])[0][k]
    pv = O.to_monty(np.array([12345, 5, 6, 7]))
    alpha_pows = O.rand_field(rng, (max(1, chip["n_constraints"]), 4))    # any table: the kernel only indexes it
    logp = max(1, (h // 2 - 1).bit_length())
    E = O.rand_field(rng, (1 << logp, 4))
    return m, k, chip, main, prep, pv, alpha_pows, E


def reference_outputs(R):
    """every reference-kernel output the tests below compare with: key -> uint32 array.  R = tests.ref_lib with oracle/_ref built, on a GPU
    (tools/gen_ref_kernels_golden.py)"""
    out = {}
    a, b = field_inputs()
    for op in ("add", "sub", "mul"):
        out[f"field/{op}"] = R.field_op(op, a, b)
    out["field/inv_nonzero"] = R.field_op("inv", a)[a != 0]
    a, b, c = ext_inputs()
    out["ext/mul"] = R.ext_op("mul", a, b)
    inv = R.ext_op("inv", a)
    out["ext/inv_of_zero"], out["ext/inv"] = inv[0], inv[4:]
    out["ext/interpolate_linear"] = R.ext_op("interpolate_linear", a, b, c)
    out["poseidon2/permute"] = R.permute(permute_inputs())
    for n_in in SPONGE_WIDTHS:
        h = R.hash_(sponge_inputs(n_in))
        out[f"sponge/hash/{n_in}"] = h
        out[f"sponge/compress/{n_in}"] = R.compress(h[:32], h[32:])
    for width, log_h in MERKLE_SHAPES:
        heap, _ = R.merkle_tree(merkle_inputs(width, log_h))
        out[f"merkle/{width}x{log_h}/layers"] = R.heap_to_layers(heap, log_h)
        # the TCS commitment wrapper (single_layer.rs:163-170): compress(root, hash([height, width])) with the reference's hash / compress
        out[f"merkle/{width}x{log_h}/commit"] = R.compress(heap[0:1], R.hash_(O.to_monty(np.array([[log_h, width]]))))[0]
    for log_h, ncols, lb in DFT_SHAPES:
        out[f"coset_dft/{log_h}/{ncols}/{lb}"] = R.batch_coset_dft(dft_inputs(log_h, ncols), lb)[0]
    out["coset_dft/max"] = R.batch_coset_dft(dft_max_inputs(), 2)[0]
    ops, vals = challenger_inputs()
    st, samples = R.challenger_script(np.zeros(34, np.uint32), ops, vals)
    out["challenger/state"], out["challenger/samples"] = st, samples[ops != 0]
    for bits in GRIND_BITS:
        out[f"grind/{bits}"] = np.array([R.grind(grind_inputs(bits).st, bits)[0]], np.uint32)
    mat, coeffs = batch_inputs()
    out["batch"] = R.batch(mat, coeffs)[0]
    vals, beta = fold_inputs()
    out["fold_mle"] = R.fold_mle_ext(vals, beta)
    out["fix_last_variable"] = R.fix_last_variable_ext(vals, beta)
    for n_vars in LAGRANGE_VARS:
        out[f"partial_lagrange/{n_vars}"] = R.partial_lagrange_ext(lagrange_inputs(n_vars))
    for wl, name, h in GKR_CHIPS:
        m, k, main, prep, alpha, betas = gkr_inputs(wl, name, h)
        chips, off = R.parse_chip_words(m["blob"])
        num, den = R.gkr_populate(R.parse_interactions(m["blob"], off, len(chips))[k], main, prep, alpha, betas)
        out[f"gkr_populate/{wl}/{name}/{h}/num"], out[f"gkr_populate/{wl}/{name}/{h}/den"] = num, den
    for wl, name, h in ZEROCHECK_CHIPS:
        m, k, chip, main, prep, pv, alpha_pows, E = zerocheck_inputs(wl, name, h)
        out[f"zerocheck/{wl}/{name}/{h}"] = R.zerocheck_node_sums(chip, main, prep, pv, alpha_pows, E)
    return out


# ---- the tests -------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    from sp1_b200 import Lib
    L = Lib(device=0)
    yield L
    L.close()


def test_field_ops_reference_vs_oracle_vs_product():
    a, b = field_inputs()
    n = a.size
    L = O.lib()
    from tests import hostcheck_lib
    P = hostcheck_lib.load()
    for op, f in (("add", L.orc_add), ("sub", L.orc_sub), ("mul", L.orc_mul)):
        exp = np.array([f(int(x), int(y)) for x, y in zip(a, b)], np.uint32)
        assert same_as_ref(f"field/{op}", exp), op
    nz = a != 0
    exp_inv = np.array([L.orc_inv(int(x)) for x in a[nz]], np.uint32)
    assert same_as_ref("field/inv_nonzero", exp_inv)
    # the product's device arithmetic sources (kb31.cuh, executed on the host by the hostcheck hooks)
    add, sub, mul = np.zeros(n, np.uint32), np.zeros(n, np.uint32), np.zeros(n, np.uint32)
    P.sp1b200_hostcheck_field(O.ptr(a), O.ptr(b), O.ptr(add), O.ptr(sub), O.ptr(mul), C.c_uint64(n))
    assert same_as_ref("field/add", add) and same_as_ref("field/sub", sub) and same_as_ref("field/mul", mul)


def test_ext_ops_reference_vs_oracle_vs_product():
    a, b, c = ext_inputs()
    n = a.shape[0]
    L = O.lib()
    from tests import hostcheck_lib
    P = hostcheck_lib.load()
    exp = np.zeros_like(a)
    for i in range(n):
        L.orc_ext_mul(O.ptr(a[i]), O.ptr(b[i]), O.ptr(exp[i]))
    assert same_as_ref("ext/mul", exp)
    got = np.zeros_like(a)
    P.sp1b200_hostcheck_ext_mul(O.ptr(a), O.ptr(b), O.ptr(got), C.c_uint64(n))
    assert same_as_ref("ext/mul", got)
    exp_inv = np.zeros_like(a)
    for i in range(4, n):
        L.orc_ext_inv(O.ptr(a[i]), O.ptr(exp_inv[i]))
    assert same_as_ref("ext/inv", exp_inv[4:])
    assert (ref_words("ext/inv_of_zero") == 0).all()   # reference convention: reciprocal(0) = 0
    got_inv = np.zeros_like(a)
    P.sp1b200_hostcheck_ext_inv(O.ptr(a[4:]), O.ptr(got_inv[4:]), C.c_uint64(n - 4))
    assert same_as_ref("ext/inv", got_inv[4:])
    # interpolateLinear (the fix_last_variable rule of every sumcheck fold): alpha.interpolateLinear(one, zero) = zero + alpha (one - zero)
    one_minus_zero = np.array([L.orc_sub(int(x), int(y)) for x, y in zip(b.reshape(-1), c.reshape(-1))], np.uint32).reshape(n, 4)
    prod = np.zeros_like(a)
    for i in range(n):
        L.orc_ext_mul(O.ptr(a[i]), O.ptr(one_minus_zero[i]), O.ptr(prod[i]))
    il = np.array([L.orc_add(int(x), int(y)) for x, y in zip(c.reshape(-1), prod.reshape(-1))], np.uint32).reshape(n, 4)
    assert same_as_ref("ext/interpolate_linear", il)


def test_poseidon2_permute_reference_vs_oracle_vs_product(lib):
    st = permute_inputs()
    exp = np.stack([O.permute(s) for s in st])
    assert same_as_ref("poseidon2/permute", exp), "oracle permutation differs from the reference's poseidon2::KoalaBearHasher::permute"
    got = st.copy()
    lib.poseidon2_permute(got)
    assert same_as_ref("poseidon2/permute", got), "product permutation kernel differs from the reference's"


@pytest.mark.parametrize("n_in", SPONGE_WIDTHS)
def test_sponge_hash_and_compress_reference_vs_oracle(n_in):
    items = sponge_inputs(n_in)
    exp = np.stack([O.hash_(v) for v in items])
    assert same_as_ref(f"sponge/hash/{n_in}", exp)
    expc = np.stack([O.compress(a, b) for a, b in zip(exp[:32], exp[32:])])
    assert same_as_ref(f"sponge/compress/{n_in}", expc)


@pytest.mark.parametrize("width,log_h", MERKLE_SHAPES)
def test_merkle_tree_reference_vs_oracle_vs_product(lib, width, log_h):
    """leafHashPacked + per-layer compress (merkle_tree.cu:27-94, launch shapes of single_layer.rs:109-150): every digest of the tree"""
    import torch
    mat = merkle_inputs(width, log_h)
    oroot, ocommit, olayers = O.merkle_commit(mat, want_layers=True)
    assert same_as_ref(f"merkle/{width}x{log_h}/layers", olayers), "oracle Merkle digests differ from the reference kernels"
    nd = (2 << log_h) - 1
    d_layers = torch.zeros(nd * 8, dtype=torch.int32, device="cuda")
    root, commit = lib.merkle_commit(mat, width, log_h, d_layers=d_layers)
    lib.sync(); torch.cuda.synchronize()
    got = d_layers.cpu().numpy().view(np.uint32).reshape(nd, 8)
    assert same_as_ref(f"merkle/{width}x{log_h}/layers", got), "product Merkle digests differ from the reference kernels"
    assert (root == got[-1]).all() and (oroot == olayers[-1]).all()
    ref_commit = ref_words(f"merkle/{width}x{log_h}/commit")
    assert (ref_commit == commit).all() and (commit == ocommit).all()


@pytest.mark.parametrize("log_h,ncols,lb", DFT_SHAPES)
def test_batch_coset_dft_reference_vs_oracle_vs_product(lib, log_h, ncols, lb):
    """encode_batch (sp1-gpu/crates/basefold/src/encoder.rs:17-34): batch_coset_dft, shift word = 1/generator, bit-reversed output"""
    msg = dft_inputs(log_h, ncols)
    got = np.zeros((ncols, 1 << (log_h + lb)), np.uint32)
    lib.rs_encode(msg, got, ncols, log_h, lb)
    assert same_as_ref(f"coset_dft/{log_h}/{ncols}/{lb}", got), "product RS-encode differs from the reference's batch_coset_dft"
    if log_h <= 16:
        assert same_as_ref(f"coset_dft/{log_h}/{ncols}/{lb}", O.rs_encode(msg, lb)), "oracle RS-encode differs from the reference's batch_coset_dft"


def test_batch_coset_dft_max_size(lib):
    """lg 21 -> 23: one full stacked column of a core shard"""
    msg = dft_max_inputs()
    got = np.zeros((1, 1 << 23), np.uint32)
    lib.rs_encode(msg, got, 1, 21, 2)
    assert same_as_ref("coset_dft/max", got)


def test_challenger_reference_device_vs_oracle_vs_product():
    """the reference's device DuplexChallenger (challenger.cuh:22-112) driven by a random transcript script"""
    from sp1_b200.lib import HostChallenger
    ops, vals = challenger_inputs()
    och, hch = O.Challenger(), HostChallenger()
    osamp, hsamp = [], []
    for i in range(ops.size):
        if ops[i] == 0:
            och.observe(vals[i:i + 1]); hch.observe(vals[i:i + 1])
        elif ops[i] == 1:
            osamp.append(och.sample(1)[0]); hsamp.append(hch.sample(1)[0])
        else:
            osamp.append(och.sample_bits(int(vals[i]))); hsamp.append(hch.sample_bits(int(vals[i])))
    assert same_as_ref("challenger/samples", np.array(osamp, np.uint32)) and same_as_ref("challenger/samples", np.array(hsamp, np.uint32))
    # final states: sponge words and buffer sizes (the device keeps stale words beyond the buffer lengths, as the 34-word format allows)
    st_ref = ref_words("challenger/state")
    for st in (och.st, hch.st):
        assert (st[:16] == st_ref[:16]).all() and st[32] == st_ref[32] and st[33] == st_ref[33]
        assert (st[16:16 + st[32]] == st_ref[16:16 + st_ref[32]]).all() and (st[24:24 + st[33]] == st_ref[24:24 + st_ref[33]]).all()


@pytest.mark.parametrize("bits", GRIND_BITS)
def test_grind_reference_kernel_witness_is_accepted(lib, bits):
    """grindKernel returns ANY valid witness (racing found_flag); the product returns the minimum one.  Both must pass
    check_witness on the oracle and the product host challenger, the product's must be <= the reference's, and replaying the
    reference's witness leaves oracle and product challengers in the same state."""
    from sp1_b200.lib import HostChallenger
    ch = grind_inputs(bits)
    w_ref = int(ref_words(f"grind/{bits}")[0])
    a, b = ch.clone(), HostChallenger(ch.st.copy())
    assert a.check_witness(bits, w_ref) and b.check_witness(bits, w_ref)
    assert (a.st == b.st).all()
    w_min, st = lib.grind(ch.st, bits)
    assert O.from_monty(np.array([w_min]))[0] <= O.from_monty(np.array([w_ref]))[0]
    c = ch.clone()
    assert c.check_witness(bits, w_min) and (c.st == st).all()


def test_batch_kernel_reference_vs_oracle():
    mat, coeffs = batch_inputs()
    width, height = mat.shape
    exp = np.zeros((height, 4), np.uint32)
    O.lib().orc_batch_columns(O.ptr(mat), C.c_uint64(width), C.c_uint64(height), O.ptr(coeffs), O.ptr(exp))
    assert same_as_ref("batch", exp)


def test_fold_and_fix_last_variable_reference_vs_oracle():
    vals, beta = fold_inputs()
    m = vals.shape[0] // 2
    exp = np.zeros((m, 4), np.uint32)
    O.lib().orc_fold_ext(O.ptr(vals), C.c_uint64(m), O.ptr(beta), 0, O.ptr(exp))
    assert same_as_ref("fold_mle", exp)
    O.lib().orc_fold_ext(O.ptr(vals), C.c_uint64(m), O.ptr(beta), 1, O.ptr(exp))
    assert same_as_ref("fix_last_variable", exp)


@pytest.mark.parametrize("n_vars", LAGRANGE_VARS)
def test_partial_lagrange_reference_vs_oracle(n_vars):
    """eq-table bit order (first coordinate = most significant bit), mle.cu:112-126 vs multilinear/src/lagrange.rs:19-45"""
    point = lagrange_inputs(n_vars)
    exp = np.zeros((1 << n_vars, 4), np.uint32)
    O.lib().orc_partial_lagrange(O.ptr(point), C.c_uint64(n_vars), O.ptr(exp))
    assert same_as_ref(f"partial_lagrange/{n_vars}", exp)


@pytest.mark.parametrize("workload,chip_name,h", GKR_CHIPS)
def test_gkr_interaction_values_reference_kernel_vs_oracle(workload, chip_name, h):
    """populateLastCircuitLayer / interactionValue (sys/lib/logup_gkr/tracegen.cu:20-160) on a calibrated chip's interactions (4-9 values,
    linear combinations of columns, preprocessed columns, constant and column multiplicities, sends and receives): numerator =
    multiplicity (negated for receives), denominator = alpha + betas[0] arg_index + sum_j betas[j+1] value_j - exactly the oracle's
    first GKR layer (crates/hypercube/src/logup_gkr/execution.rs:13-36 restated)"""
    m, k, main, prep, alpha, betas = gkr_inputs(workload, chip_name, h)
    n_inter = _ref(f"gkr_populate/{workload}/{chip_name}/{h}/num")["shape"][0]
    assert n_inter >= 4
    onum = np.zeros((n_inter, h), np.uint32); oden = np.zeros((n_inter, h, 4), np.uint32)
    prepf = np.ascontiguousarray(prep).reshape(-1) if prep is not None else np.zeros(1, np.uint32)
    n = O.lib().orc_interaction_values(O.ptr(np.ascontiguousarray(m["blob"])), C.c_uint32(k), O.ptr(np.ascontiguousarray(main).reshape(-1)), O.ptr(prepf),
                                       C.c_uint64(h), O.ptr(alpha), O.ptr(betas.reshape(-1)), C.c_uint32(betas.shape[0]), O.ptr(onum.reshape(-1)),
                                       O.ptr(oden.reshape(-1)))
    assert n == n_inter
    assert same_as_ref(f"gkr_populate/{workload}/{chip_name}/{h}/num", onum), "LogUp numerators (multiplicities) differ from the reference kernel"
    assert same_as_ref(f"gkr_populate/{workload}/{chip_name}/{h}/den", oden), "LogUp denominators differ from the reference kernel"


@pytest.mark.parametrize("workload,chip_name,h", ZEROCHECK_CHIPS)
def test_zerocheck_interpreter_reference_kernel_vs_oracle(workload, chip_name, h):
    """zerocheck_fused_sequential<felt_t, 1024> (sys/lib/zerocheck/sequential.cu:49-190): the reference's own bytecode interpreter run on
    this repository's chip programs (DagInstr / LeafRef / assert tables in the reference layout): opcode semantics, leaf sources,
    public values, alpha-index lookup, node interpolation {0, 2, 4} and the eq weighting give the oracle's round-0 node sums"""
    m, k, chip, main, prep, pv, alpha_pows, E = zerocheck_inputs(workload, chip_name, h)
    ref = ref_words(f"zerocheck/{workload}/{chip_name}/{h}")
    exp = np.zeros(12, np.uint32)
    prepf = np.ascontiguousarray(prep).reshape(-1) if prep is not None else np.zeros(1, np.uint32)
    rc = O.lib().orc_zerocheck_node_sums(O.ptr(np.ascontiguousarray(m["blob"])), C.c_uint32(k), O.ptr(np.ascontiguousarray(main).reshape(-1)), O.ptr(prepf),
                                         C.c_uint64(h), O.ptr(pv), C.c_uint32(pv.size), O.ptr(alpha_pows.reshape(-1)), O.ptr(E.reshape(-1)), O.ptr(exp))
    assert rc == 0
    assert (ref.reshape(-1) == exp).all(), "constraint interpreter node sums differ from the reference kernel"
    assert ref.any()
