// mock_circuit.cpp — the reference's own circuit proved through the C++ host layer (include/pb200.hpp).
//
// Restates, call for call, /root/reference/src/zk/gadgets.rs `maybe_equal` (:49-84), `scalar_decomposition_gadget`
// (:186-225), `min_bound` (:120-145) and /root/reference/src/zk/circuits.rs `MockCircuit::valid_balance` (:51-60) over
// pb200::StandardComposer, then runs preprocess → prove on the GPU and verify on the host, plus an EvaluationDomain round
// trip and a KZG commit.  Exit code 0 = everything checked.  Built by `make -C plonk-prototype_b200/csrc example`.
#include <cstdio>

#include "../include/pb200.hpp"

using namespace pb200;

struct AllocatedScalar {  // allocated_scalar.rs:25-38
    Variable var;
    BlsScalar scalar;
    static AllocatedScalar allocate(StandardComposer &c, const BlsScalar &s) { return {c.add_input(s), s}; }
};

static Variable maybe_equal(StandardComposer &c, const AllocatedScalar &a, const AllocatedScalar &b) {
    const Variable u = c.add({BlsScalar::one(), a.var}, {-BlsScalar::one(), b.var}, BlsScalar::zero());
    const auto inv = (a.scalar - b.scalar).invert();
    const Variable z = c.add_input(inv.first ? inv.second : BlsScalar::zero());
    const Variable y = c.mul(-BlsScalar::one(), z, u, BlsScalar::one());
    c.mul_gate(y, u, u, BlsScalar::one(), BlsScalar::zero(), BlsScalar::zero());
    return y;
}

static Variable scalar_decomposition_gadget(StandardComposer &c, size_t num_bits, const AllocatedScalar &witness) {
    const auto bytes = witness.scalar.to_bytes();
    std::vector<Variable> bit_vars;
    std::vector<uint8_t> bits(256);
    for (int i = 0; i < 256; i++) {
        bits[i] = (bytes[i / 8] >> (i % 8)) & 1;
        bit_vars.push_back(c.add_input(BlsScalar::from(bits[i])));  // all 256 are allocated, the first num_bits used
    }
    AllocatedScalar acc{c.add_witness_to_circuit_description(BlsScalar::zero()), BlsScalar::zero()};
    for (size_t power = 0; power < num_bits; power++) {
        c.boolean_gate(bit_vars[power]);
        const BlsScalar two_pow = BlsScalar::from(2).pow(power);
        acc.var = c.add({two_pow, bit_vars[power]}, {BlsScalar::one(), acc.var}, BlsScalar::zero());
        acc.scalar = acc.scalar + two_pow * BlsScalar::from(bits[power]);
    }
    return maybe_equal(c, acc, witness);
}

static Variable min_bound(StandardComposer &c, const BlsScalar &min_range, const AllocatedScalar &witness, size_t num_bits) {
    const Variable v = c.add({BlsScalar::one(), witness.var}, {BlsScalar::zero(), witness.var}, -min_range);
    return scalar_decomposition_gadget(c, num_bits, AllocatedScalar{v, witness.scalar - min_range});
}

#define CHECK(cond)                                                    \
    do {                                                               \
        if (!(cond)) {                                                 \
            fprintf(stderr, "FAILED: %s (line %d)\n", #cond, __LINE__); \
            return 1;                                                  \
        }                                                              \
    } while (0)

int main() {
    try {
        Context ctx(0);
        const std::string label = "manta-mock-circuit";
        const BlsScalar tau = BlsScalar::from(0x7e57c0de);

        // MockCircuit::valid_balance: note value 1 000 000 covers tx 900 000 + gas 21 000
        Prover prover = Prover::new_(ctx, label);
        StandardComposer &cs = prover.mut_cs();
        const AllocatedScalar note = AllocatedScalar::allocate(cs, BlsScalar::from(1000000));
        const Variable out = min_bound(cs, BlsScalar::from(900000) + BlsScalar::from(21000), note, 30);
        CHECK(cs.value_of(out) == BlsScalar::one());
        const BlsScalar minus_one = -BlsScalar::one();
        cs.constrain_to_constant(out, BlsScalar::zero(), &minus_one);  // expose the 0/1 result as a public input
        CommitKey ck = CommitKey::setup(ctx, 1023, tau);  // PublicParameters::setup(max_degree): covers the circuit and the commits below
        prover.preprocess(ck);
        const ProofBytes proof = prover.prove(ck);
        CHECK(proof == prover.prove(ck));  // deterministic (no blinding in 0.8.x)
        CHECK(verify_proof(prover.verifier_key(), prover.padded_size(), label, proof, cs.public_inputs_sparse_store(), tau));
        std::map<uint32_t, BlsScalar> wrong = cs.public_inputs_sparse_store();
        wrong.begin()->second = BlsScalar::zero();
        CHECK(!verify_proof(prover.verifier_key(), prover.padded_size(), label, proof, wrong, tau));
        ProofBytes tampered = proof;
        tampered[600] ^= 1;
        CHECK(!verify_proof(prover.verifier_key(), prover.padded_size(), label, tampered, cs.public_inputs_sparse_store(), tau));
        {  // the valid and the two invalid cases above, verified in one batch on the GPU
            const std::array<uint8_t, 32> seed{0x5e, 0xed};
            const std::vector<bool> verdicts = verify_proofs(ctx, prover.verifier_key(), prover.padded_size(), label, {proof, proof, tampered},
                                                             {cs.public_inputs_sparse_store(), wrong, cs.public_inputs_sparse_store()}, tau, seed);
            CHECK(verdicts == std::vector<bool>({true, false, false}));
        }

        // MockCircuit::prove_ownership (/root/reference/src/zk/circuits.rs:63-66): sk·G computed in circuit by the fixed-base
        // widget equals the public key, which enters as two public inputs
        {
            Prover own = Prover::new_(ctx, "manta-prove-ownership");
            StandardComposer &c2 = own.mut_cs();
            const BlsScalar sk = BlsScalar::from(0x0A11CE5EC2E7ull);
            const jubjub::Affine pk_point = jubjub::mul(jubjub::generator(), sk.reduce());
            const Point circuit_pk = c2.fixed_base_scalar_mul(c2.add_input(sk), jubjub::generator());
            c2.assert_equal_public_point(circuit_pk, pk_point);
            own.preprocess(ck);
            const ProofBytes p2 = own.prove(ck);
            CHECK(verify_proof(own.verifier_key(), own.padded_size(), "manta-prove-ownership", p2, c2.public_inputs_sparse_store(), tau));
            std::map<uint32_t, BlsScalar> other_key = c2.public_inputs_sparse_store();
            other_key.begin()->second = other_key.begin()->second + BlsScalar::one();
            CHECK(!verify_proof(own.verifier_key(), own.padded_size(), "manta-prove-ownership", p2, other_key, tau));
        }

        // EvaluationDomain round trips and the error rule
        EvaluationDomain dom = EvaluationDomain::new_(ctx, 1000);
        CHECK(dom.size() == 1024);
        std::vector<BlsScalar> poly;
        for (uint64_t i = 0; i < 1000; i++) poly.push_back(BlsScalar::from(i * i + 7));
        std::vector<BlsScalar> back = dom.coset_ifft(dom.coset_fft(poly));
        for (size_t i = 0; i < 1024; i++) CHECK(back[i] == (i < 1000 ? poly[i] : BlsScalar::zero()));
        bool threw = false;
        try {
            EvaluationDomain::new_(ctx, ((size_t)1 << 31) + 1);
        } catch (const InvalidEvalDomainSize &) {
            threw = true;
        }
        CHECK(threw);

        // commit(p) + commit(q) and commit(p + q) encode the same point when doubled scalars are used: commit(2p) = commit(p + p)
        std::vector<BlsScalar> twice;
        for (const auto &c : poly) twice.push_back(c + c);
        const G1Projective c1 = ck.commit(poly), c2 = ck.commit(twice);
        CHECK(!c1.is_identity() && !c2.is_identity() && c1.to_bytes() != c2.to_bytes());
        CHECK(ck.commit(std::vector<BlsScalar>(10)).is_identity());  // the zero polynomial commits to the identity
        printf("mock_circuit ok: %zu gates (padded %zu), proof verified, tampering rejected\n", cs.circuit_size(), prover.padded_size());
        return 0;
    } catch (const std::exception &e) {
        fprintf(stderr, "error: %s\n", e.what());
        return 2;
    }
}
