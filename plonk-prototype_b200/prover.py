"""Host-side mirror of the dusk-plonk 0.8.2 proving API the reference's circuits are written against
(`StandardComposer`, `Prover`, `PublicParameters`; crate pinned at /root/reference/Cargo.toml:19; the composer
calls mirrored here are exactly the ones /root/reference/src/zk/gadgets.rs:60-81,132,165,206-218 and
circuits.rs:57,71 make — SURVEY.md App. C).

Circuit synthesis is host-side bookkeeping in the reference too (it only appends rows to the composer's
vectors), so it stays on the host here: Python ints for the witness values, numpy for the column images.
Everything after synthesis — preprocessing and the five prover rounds — runs on the GPU behind
`pb200_preprocess` / `pb200_prove` (csrc/plonk.cu).  There is no CPU proving path.
"""
import numpy as np

from . import _native
from .domain import default_context

R = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
_MONT = (1 << 256) % R
SELECTORS = ("q_m", "q_l", "q_r", "q_o", "q_c", "q_4", "q_arith", "q_range", "q_logic", "q_fixed_group_add",
             "q_variable_group_add")


def scalars_to_mont(values):
    """Python ints (canonical, any sign) → (n, 4) uint64 Montgomery limbs, the ABI's scalar image."""
    buf = b"".join(((v % R) * _MONT % R).to_bytes(32, "little") for v in values)
    return np.frombuffer(buf, dtype="<u8").reshape(-1, 4).copy()


class StandardComposer:
    """Gate equation q_arith·(q_m·a·b + q_l·a + q_r·b + q_o·c + q_4·d + q_c) + PI = 0 (SURVEY.md App. B.3)."""

    def __init__(self):
        self.q = {k: [] for k in SELECTORS}
        self.w_l, self.w_r, self.w_o, self.w_4 = [], [], [], []
        self.variables = []                 # Variable index → BlsScalar value (Python int)
        self.public_inputs_sparse_store = {}
        self.n = 0
        self.zero_var = 0
        self.zero_var = self.add_witness_to_circuit_description(0)
        self.add_dummy_constraints()

    def circuit_size(self):
        return self.n

    # ---- allocation
    def add_input(self, s):
        self.variables.append(s % R)
        return len(self.variables) - 1

    def _row(self, a, b, c, d, q_m=0, q_l=0, q_r=0, q_o=0, q_c=0, q_4=0, q_arith=1, q_range=0, pi=None, q_logic=0,
             q_fixed_group_add=0, q_variable_group_add=0):
        row = dict(q_m=q_m, q_l=q_l, q_r=q_r, q_o=q_o, q_c=q_c, q_4=q_4, q_arith=q_arith, q_range=q_range, q_logic=q_logic,
                   q_fixed_group_add=q_fixed_group_add, q_variable_group_add=q_variable_group_add)
        for k in SELECTORS:
            self.q[k].append(row.get(k, 0) % R)
        self.w_l.append(a)
        self.w_r.append(b)
        self.w_o.append(c)
        self.w_4.append(d)
        if pi is not None:
            self.public_inputs_sparse_store[self.n] = pi % R
        self.n += 1

    # ---- the calls the reference's gadgets make
    def poly_gate(self, a, b, c, q_m, q_l, q_r, q_o, q_c, pi=None):
        self._row(a, b, c, self.zero_var, q_m=q_m, q_l=q_l, q_r=q_r, q_o=q_o, q_c=q_c, pi=pi)
        return a, b, c

    def add(self, q_l_a, q_r_b, q_c, pi=None):
        (q_l, a), (q_r, b) = q_l_a, q_r_b
        c = self.add_input(q_l * self.variables[a] + q_r * self.variables[b] + q_c + (pi or 0))
        self._row(a, b, c, self.zero_var, q_l=q_l, q_r=q_r, q_o=-1, q_c=q_c, pi=pi)
        return c

    def mul(self, q_m, a, b, q_c, pi=None):
        c = self.add_input(q_m * self.variables[a] * self.variables[b] + q_c + (pi or 0))
        self._row(a, b, c, self.zero_var, q_m=q_m, q_o=-1, q_c=q_c, pi=pi)
        return c

    def add_gate(self, a, b, c, q_l, q_r, q_o, q_c, pi=None):
        self._row(a, b, c, self.zero_var, q_l=q_l, q_r=q_r, q_o=q_o, q_c=q_c, pi=pi)
        return c

    def mul_gate(self, a, b, c, q_m, q_o, q_c, pi=None):
        self._row(a, b, c, self.zero_var, q_m=q_m, q_o=q_o, q_c=q_c, pi=pi)
        return c

    def boolean_gate(self, a):
        self._row(a, a, a, self.zero_var, q_m=1, q_o=-1)
        return a

    def constrain_to_constant(self, a, constant, pi=None):
        self._row(a, a, a, self.zero_var, q_l=1, q_c=-constant, pi=pi)

    def assert_equal(self, a, b):
        self._row(a, b, self.zero_var, self.zero_var, q_l=1, q_r=-1)

    def add_witness_to_circuit_description(self, value):
        var = self.add_input(value)
        self.constrain_to_constant(var, value, None)
        return var

    def range_rows(self, a, b, c, d):
        """One row of the range widget (q_range = 1): quads c−4d, b−4c, a−4b, d_next−4a ∈ {0,1,2,3}."""
        self._row(a, b, c, d, q_arith=0, q_range=1)

    def big_add(self, q_l_a, q_r_b, q_4_d, q_c, pi=None):
        """`big_add((q_l, a), (q_r, b), Some((q_4, d)), q_c, pi) -> Variable`: allocates c = q_l·a + q_r·b + q_4·d + q_c + pi."""
        (q_l, a), (q_r, b) = q_l_a, q_r_b
        q_4, d = q_4_d if q_4_d is not None else (0, self.zero_var)
        c = self.add_input(q_l * self.variables[a] + q_r * self.variables[b] + q_4 * self.variables[d] + q_c + (pi or 0))
        self._row(a, b, c, d, q_l=q_l, q_r=q_r, q_o=-1, q_4=q_4, q_c=q_c, pi=pi)
        return c

    def big_add_gate(self, a, b, c, d, q_l, q_r, q_o, q_4, q_c, pi=None):
        self._row(a, b, c, self.zero_var if d is None else d, q_l=q_l, q_r=q_r, q_o=q_o, q_4=q_4, q_c=q_c, pi=pi)
        return c

    # ---- constraint_system::ecc — points are (x, y) pairs of variables on JubJub (plonk-prototype_b200/jubjub.py)
    def fixed_base_scalar_mul(self, jubjub_scalar, generator):
        """`fixed_base_scalar_mul(scalar, generator) -> Point` (/root/reference/src/zk/gadgets.rs:34,37; circuits.rs:64):
        a 256-step ladder over the 2-bit windowed NAF of the scalar, most significant digit first.  Row i holds the point
        accumulator (w_l, w_r), x_α·y_α of the point added (w_o) and the scalar accumulator (w_4), with the generator
        multiple 2^(255−i)·G in q_l, q_r, q_c and q_fixed_group_add = 1; one plain row carries the final accumulators."""
        from . import jubjub as jj
        num_bits = 256
        multiples = [tuple(generator)]
        for _ in range(num_bits - 1):
            multiples.append(jj.add(multiples[-1], multiples[-1]))
        multiples.reverse()
        k = self.variables[jubjub_scalar]
        if k >= jj.JJ_ORDER:
            raise ValueError("fixed_base_scalar_mul: the scalar is not a canonical JubJub scalar")  # JubJubScalar::from_bytes(..).unwrap()
        scalar_acc, point_acc, xy_alphas = [0], [jj.IDENTITY], []
        for i, entry in enumerate(reversed(jj.wnaf2(k))):
            to_add = jj.IDENTITY if entry == 0 else (multiples[i] if entry == 1 else jj.neg(multiples[i]))
            scalar_acc.append((2 * scalar_acc[i] + entry) % R)
            point_acc.append(jj.add(point_acc[i], to_add))
            xy_alphas.append(to_add[0] * to_add[1] % R)
        for i in range(num_bits):
            acc_x, acc_y = self.add_input(point_acc[i][0]), self.add_input(point_acc[i][1])
            accumulated_bit = self.add_input(scalar_acc[i])
            if i == 0:
                self.constrain_to_constant(acc_x, 0, None)
                self.constrain_to_constant(acc_y, 1, None)
                self.constrain_to_constant(accumulated_bit, 0, None)
            x_beta, y_beta = multiples[i]
            xy_alpha = self.add_input(xy_alphas[i])
            self._row(acc_x, acc_y, xy_alpha, accumulated_bit, q_l=x_beta, q_r=y_beta, q_c=x_beta * y_beta, q_arith=0,
                      q_fixed_group_add=1)
        acc_x, acc_y = self.add_input(point_acc[num_bits][0]), self.add_input(point_acc[num_bits][1])
        last_accumulated_bit = self.add_input(scalar_acc[num_bits])
        self.big_add_gate(acc_x, acc_y, self.zero_var, last_accumulated_bit, 0, 0, 0, 0, 0, None)
        self.assert_equal(last_accumulated_bit, jubjub_scalar)
        return (acc_x, acc_y)

    def point_addition_gate(self, point_a, point_b):
        """`point_addition_gate(p1, p2) -> Point` (/root/reference/src/zk/gadgets.rs:40): two rows, the first with
        q_variable_group_add = 1 holding (x1, y1, x2, y2), the second (x3, y3, 0, x1·y2)."""
        from . import jubjub as jj
        (x1, y1), (x2, y2) = point_a, point_b
        v = self.variables
        x3v, y3v = jj.add((v[x1], v[y1]), (v[x2], v[y2]))
        x1_y2 = self.add_input(v[x1] * v[y2])
        x3, y3 = self.add_input(x3v), self.add_input(y3v)
        self._row(x1, y1, x2, y2, q_arith=0, q_variable_group_add=1)
        self._row(x3, y3, self.zero_var, x1_y2, q_arith=0)
        return (x3, y3)

    def assert_equal_public_point(self, point, public_point):
        """`assert_equal_public_point` (/root/reference/src/zk/circuits.rs:65): two public-input constraints."""
        self.constrain_to_constant(point[0], 0, -public_point[0])
        self.constrain_to_constant(point[1], 0, -public_point[1])

    # ---- constraint_system::logic — XOR / AND of two num_bits-bit variables, one 2-bit quad per row from the top
    def _logic_gate(self, a, b, num_bits, is_xor):
        assert num_bits % 2 == 0
        av, bv = self.variables[a], self.variables[b]
        nq, sel = num_bits // 2, (-1 if is_xor else 1)
        rows_l, rows_r, rows_4, rows_o = [self.zero_var], [self.zero_var], [self.zero_var], []
        la = ra = oa = 0
        for i in range(nq):
            sh = 2 * (nq - 1 - i)
            lq, rq = (av >> sh) & 3, (bv >> sh) & 3
            oq = (lq ^ rq) if is_xor else (lq & rq)
            la, ra, oa = 4 * la + lq, 4 * ra + rq, 4 * oa + oq
            rows_l.append(self.add_input(la))
            rows_r.append(self.add_input(ra))
            rows_4.append(self.add_input(oa))
            rows_o.append(self.add_input(lq * rq))
        rows_o.append(self.zero_var)
        for i in range(nq + 1):
            last = i == nq
            self._row(rows_l[i], rows_r[i], rows_o[i], rows_4[i], q_arith=0, q_c=0 if last else sel, q_logic=0 if last else sel)
        self.assert_equal(a, rows_l[nq])
        self.assert_equal(b, rows_r[nq])
        return rows_4[nq]

    def xor_gate(self, a, b, num_bits):
        return self._logic_gate(a, b, num_bits, True)

    def and_gate(self, a, b, num_bits):
        return self._logic_gate(a, b, num_bits, False)

    def add_dummy_constraints(self):
        six, one, seven, m20 = (self.add_input(v) for v in (6, 1, 7, -20))
        self._row(six, seven, m20, one, q_m=1, q_l=2, q_r=3, q_o=4, q_c=4, q_4=1)
        self._row(m20, six, seven, self.zero_var, q_m=1, q_l=1, q_r=1, q_o=1, q_c=127)

    # ---- column images for the ABI
    def selector_columns(self):
        out = []
        for k in SELECTORS:
            col = self.q[k]
            out.append(scalars_to_mont(col) if any(col) else None)
        return out

    def wire_columns(self):
        return [np.asarray(w, dtype=np.uint32) for w in (self.w_l, self.w_r, self.w_o, self.w_4)]


class PublicParameters:
    """`PublicParameters::setup(max_degree, rng)` with the trapdoor supplied by the caller (test / benchmark SRS):
    powers_of_g[i] = τ^i·G generated on the device and kept resident, pre-doubled window copies for fast commits."""

    def __init__(self, max_degree, tau, ctx=None, precompute=True):
        self.ctx = ctx or default_context()
        self.n_points = max_degree + 1
        self.srs = self.ctx.srs_generate(scalars_to_mont([tau]), self.n_points)
        if precompute and self.n_points <= (1 << 22):
            self.ctx.srs_precompute(self.srs)

        self.beta_h = _native.opening_key_from_tau(scalars_to_mont([tau]))   # the opening key's β·H (G and H are the generators)

    def to_raw_bytes(self):
        """`PublicParameters::to_raw_bytes`: opening key (240 bytes) ‖ commit key (memory image of the points) — serial.py."""
        from . import serial
        return serial.opening_key_to_bytes(self.beta_h) + serial.commit_key_to_raw_bytes(self.ctx, self.srs)

    @classmethod
    def from_slice_unchecked(cls, data, ctx=None, precompute=True):
        """`PublicParameters::from_slice_unchecked`: parameters cached with `to_raw_bytes` back onto the GPU."""
        from . import serial
        self = cls.__new__(cls)
        self.ctx = ctx or default_context()
        self.beta_h = serial.opening_key_from_bytes(bytes(data[:serial.OPENING_KEY_SIZE]))
        self.srs = serial.commit_key_from_slice_unchecked(self.ctx, bytes(data[serial.OPENING_KEY_SIZE:]), precompute)
        self.n_points = _native.lib().pb200_srs_len(self.srs)
        return self

    def to_var_bytes(self):
        """`PublicParameters::to_var_bytes`: opening key (240 bytes) ‖ commit key as 48-byte compressed points (encoded on
        the GPU) — the distributable form, e.g. of a setup ceremony's output."""
        from . import serial
        return serial.opening_key_to_bytes(self.beta_h) + serial.commit_key_to_var_bytes(self.ctx, self.srs)

    @classmethod
    def from_slice(cls, data, ctx=None, precompute=True):
        """`PublicParameters::from_slice`: parameters in the to_var_bytes form, checked.  β·H must be a point of G2 (host);
        every commit-key point is decoded and checked on the GPU (flags, x < p, on the curve, prime-order subgroup).
        ValueError on anything invalid; nothing stays allocated then."""
        from . import serial
        self = cls.__new__(cls)
        self.ctx = ctx or default_context()
        self.beta_h = serial.opening_key_from_bytes_checked(bytes(data[:serial.OPENING_KEY_SIZE]))
        self.srs = serial.commit_key_from_slice(self.ctx, bytes(data[serial.OPENING_KEY_SIZE:]), precompute)
        self.n_points = _native.lib().pb200_srs_len(self.srs)
        return self

    def close(self):
        if self.srs is not None:
            self.ctx.srs_free(self.srs)
            self.srs = None


def torch_allgather(dist, device=None):
    """The all-gather a sharded key calls between an MSM and the transcript: bytes in → world × bytes out, rank-major.
    `dist` is torch.distributed with an initialised process group (NCCL over NVLink on the GPU box — `device` is then
    this rank's cuda device — or gloo in the CPU tests)."""
    import torch

    def gather(send):
        t = torch.frombuffer(bytearray(send), dtype=torch.uint8)
        if device is not None:
            t = t.to(device)
        out = torch.empty(dist.get_world_size() * t.numel(), dtype=torch.uint8, device=t.device)
        dist.all_gather_into_tensor(out, t)
        return out.cpu().numpy().tobytes()

    return gather


def torch_device_collectives(dist, device):
    """(alltoall_dev, allgather_dev) for a sharded key: NCCL collectives on raw device pointers of the library's buffers,
    wrapped as torch tensors through __cuda_array_interface__ (no copy).  Both return after the collective has completed."""
    import torch

    class _Dev:
        def __init__(self, ptr, nbytes):
            self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (int(ptr), False), "version": 3}

    def view(ptr, nbytes):
        return torch.as_tensor(_Dev(ptr, nbytes), device=device)

    def alltoall(send, recv, bytes_per_peer):
        world = dist.get_world_size()
        dist.all_to_all_single(view(recv, world * bytes_per_peer), view(send, world * bytes_per_peer))
        torch.cuda.synchronize(device)

    def allgather(send, recv, nbytes):
        dist.all_gather_into_tensor(view(recv, dist.get_world_size() * nbytes), view(send, nbytes))
        torch.cuda.synchronize(device)

    return alltoall, allgather


class ShardedParameters:
    """This rank's slice powers_of_g[rank·n/world .. (rank+1)·n/world) of `PublicParameters::setup(n − 1)`."""

    def __init__(self, n_points, tau, rank, world, ctx=None, precompute=True):
        assert n_points % world == 0
        self.ctx = ctx or default_context()
        self.n_points, self.rank, self.world = n_points, rank, world
        per = n_points // world
        self.srs = self.ctx.srs_generate_range(scalars_to_mont([tau]), rank * per, per)
        if precompute and per <= (1 << 22):
            self.ctx.srs_precompute(self.srs)

    def close(self):
        if self.srs is not None:
            self.ctx.srs_free(self.srs)
            self.srs = None


class Prover:
    """`Prover::new(label)`, `.mut_cs()`, `.preprocess(&ck)`, `.prove(&ck)`."""

    def __init__(self, label, ctx=None):
        self.label = bytes(label)
        self.cs = StandardComposer()
        self.ctx = ctx or default_context()
        self._pk = None
        self.verifier_key_bytes = None

    def mut_cs(self):
        return self.cs

    def circuit_size(self):
        return self.cs.circuit_size()

    def preprocess(self, pp):
        if self._pk is not None:
            raise RuntimeError("CircuitAlreadyPreprocessed")
        self._pk, self.verifier_key_bytes = self.ctx.preprocess(pp.srs, self.cs.selector_columns(), self.cs.wire_columns(),
                                                                len(self.cs.variables), self.label)
        self.padded_size = self.ctx.prover_key_size(self._pk)

    def prove(self, pp, variables=None):
        """Returns `Proof::to_bytes()` (1040 bytes).  `variables` overrides the composer's assignment (same circuit,
        new witness) as (n_vars, 4) Montgomery limbs."""
        if self._pk is None:
            self.preprocess(pp)
        vals = variables if variables is not None else scalars_to_mont(self.cs.variables)
        pis = sorted(self.cs.public_inputs_sparse_store.items())
        pos = np.asarray([p for p, _ in pis], dtype=np.uint32)
        piv = scalars_to_mont([v for _, v in pis]) if pis else np.zeros((0, 4), np.uint64)
        return self.ctx.prove(pp.srs, self._pk, vals, pos, piv)

    def close(self):
        if self._pk is not None:
            self.ctx.prover_key_free(self._pk)
            self._pk = None
