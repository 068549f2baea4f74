//go:build b200

package b200

/*
#include "b200g16.h"
*/
import "C"

import (
	"errors"
	"runtime"
	"unsafe"

	curve "github.com/consensys/gnark-crypto/ecc/bn254"
	"github.com/consensys/gnark-crypto/ecc/bn254/fr"
	"github.com/consensys/gnark-crypto/ecc/bn254/fr/fft"
	"github.com/consensys/gnark-crypto/ecc/bn254/fr/pedersen"
	groth16_bn254 "github.com/consensys/gnark/backend/groth16/bn254"
	"github.com/consensys/gnark/constraint"
	cs "github.com/consensys/gnark/constraint/bn254"
)

// Setup has gnark's signature, groth16.Setup(ccs) at mt.go:448, and returns the same key as gnark's Setup for the same
// toxic waste: b200g16_setup runs setupABC, the K / Z scalars, the infinity filtering and every fixed-base
// multiplication on the GPU.  The toxic waste is drawn from crypto/rand, as gnark draws it.  The point vectors are
// downloaded into gnark's pk (so it serialises and works with any backend) and also stay resident: the returned
// ProvingKey proves without a second upload.  At most one BSB22 commitment, like the rest of the library.
func Setup(r1cs *cs.R1CS) (*ProvingKey, *groth16_bn254.VerifyingKey, error) {
	commitmentInfo := r1cs.CommitmentInfo.(constraint.Groth16Commitments)
	if len(commitmentInfo) > 1 {
		return nil, nil, errors.New("b200: Setup supports at most one BSB22 commitment")
	}
	nbInternal, nbSecret, nbPublic := r1cs.GetNbVariables()
	nbWires := nbInternal + nbSecret + nbPublic

	// L, R, O as CSR by constraint, straight from gnark's Term{CID, VID}
	var rows [3][]uint64
	var wires, cids [3][]uint32
	for k := range rows {
		rows[k] = append(make([]uint64, 0, r1cs.GetNbConstraints()+1), 0)
	}
	it := r1cs.GetR1CIterator()
	for c := it.Next(); c != nil; c = it.Next() {
		for k, lc := range []constraint.LinearExpression{c.L, c.R, c.O} {
			for _, t := range lc {
				wires[k] = append(wires[k], t.VID)
				cids[k] = append(cids[k], t.CID)
			}
			rows[k] = append(rows[k], uint64(len(wires[k])))
		}
	}

	var tw C.b200g16_toxic
	for _, dst := range []*[4]C.uint64_t{&tw.tau, &tw.alpha, &tw.beta, &tw.gamma, &tw.delta, &tw.sigma} {
		var e fr.Element // SetRandom draws from crypto/rand
		for e.IsZero() {
			if _, err := e.SetRandom(); err != nil {
				return nil, nil, err
			}
		}
		for i := 0; i < 4; i++ {
			dst[i] = C.uint64_t(e[i])
		}
	}

	var pin runtime.Pinner
	defer pin.Unpin()
	ptr32 := func(v []uint32) *C.uint32_t {
		if len(v) == 0 {
			return nil
		}
		pin.Pin(&v[0])
		return (*C.uint32_t)(unsafe.Pointer(&v[0]))
	}
	ptr64 := func(v []uint64) *C.uint64_t {
		pin.Pin(&v[0])
		return (*C.uint64_t)(unsafe.Pointer(&v[0]))
	}
	d := C.b200g16_r1cs_desc{
		n_constraints: C.size_t(r1cs.GetNbConstraints()), n_wires: C.size_t(nbWires), n_public: C.size_t(nbPublic),
		n_coeffs: C.size_t(len(r1cs.Coefficients)), commitment_wire: -1,
		l_row: ptr64(rows[0]), l_wire: ptr32(wires[0]), l_coeff: ptr32(cids[0]),
		r_row: ptr64(rows[1]), r_wire: ptr32(wires[1]), r_coeff: ptr32(cids[1]),
		o_row: ptr64(rows[2]), o_wire: ptr32(wires[2]), o_coeff: ptr32(cids[2]),
	}
	if len(r1cs.Coefficients) > 0 {
		pin.Pin(&r1cs.Coefficients[0])
		d.coeffs = u64(unsafe.Pointer(&r1cs.Coefficients[0]))
	}
	var committed []uint32
	var publicCommitted []int
	if len(commitmentInfo) == 1 {
		ci := commitmentInfo[0]
		for _, w := range ci.PrivateCommitted {
			committed = append(committed, uint32(w))
		}
		d.private_committed, d.n_private_committed = ptr32(committed), C.size_t(len(committed))
		d.commitment_wire = C.int64_t(ci.CommitmentIndex)
		publicCommitted = ci.PublicAndCommitmentCommitted
	}

	pk := &ProvingKey{}
	if err := call(func() C.int { return C.b200g16_init(0, &pk.ctx) }); err != nil {
		return nil, nil, err
	}
	infA, infB, kSkip := make([]byte, nbWires), make([]byte, nbWires), make([]byte, nbWires)
	pin.Pin(&infA[0])
	pin.Pin(&infB[0])
	pin.Pin(&kSkip[0])
	var out C.b200g16_setup_out
	pin.Pin(&out) // the pk desc below points into it
	if err := call(func() C.int {
		return C.b200g16_setup(pk.ctx, &d, &tw, (*C.uint8_t)(unsafe.Pointer(&infA[0])),
			(*C.uint8_t)(unsafe.Pointer(&infB[0])), (*C.uint8_t)(unsafe.Pointer(&kSkip[0])), &out)
	}); err != nil {
		C.b200g16_destroy(pk.ctx)
		return nil, nil, err
	}
	defer C.b200g16_bases_free(out.vk_k)
	// from here on the pk owns what the setup made: every error path releases it all (and the ctx) through Free
	pk.owned = []*C.b200g16_bases{out.a, out.b, out.k, out.z, out.b2}
	if len(commitmentInfo) == 1 {
		pk.pedBasis, pk.pedSigma = []*C.b200g16_bases{out.ped_basis}, []*C.b200g16_bases{out.ped_basis_exp_sigma}
	}
	fail := func(err error) (*ProvingKey, *groth16_bn254.VerifyingKey, error) {
		pk.Free()
		return nil, nil, err
	}

	g1 := func(b *C.b200g16_bases) ([]curve.G1Affine, error) {
		v := make([]curve.G1Affine, int(C.b200g16_bases_len(b)))
		if len(v) == 0 {
			return v, nil
		}
		return v, call(func() C.int {
			return C.b200g16_bases_download(b, 0, C.size_t(len(v)), u64(unsafe.Pointer(&v[0])))
		})
	}
	var err error
	n := uint64(1) << uint(out.log2_domain)
	pk.Domain = *fft.NewDomain(n)
	pk.InfinityA, pk.InfinityB = make([]bool, nbWires), make([]bool, nbWires)
	for i := range infA {
		pk.InfinityA[i], pk.InfinityB[i] = infA[i] != 0, infB[i] != 0
		pk.NbInfinityA += uint64(infA[i])
		pk.NbInfinityB += uint64(infB[i])
	}
	if pk.G1.A, err = g1(out.a); err == nil {
		if pk.G1.B, err = g1(out.b); err == nil {
			if pk.G1.K, err = g1(out.k); err == nil {
				pk.G1.Z, err = g1(out.z)
			}
		}
	}
	if err != nil {
		return fail(err)
	}
	pk.G2.B = make([]curve.G2Affine, int(C.b200g16_bases_len(out.b2)))
	if len(pk.G2.B) > 0 {
		if err := call(func() C.int {
			return C.b200g16_bases_download(out.b2, 0, C.size_t(len(pk.G2.B)), u64(unsafe.Pointer(&pk.G2.B[0])))
		}); err != nil {
			return fail(err)
		}
	}
	copyPt := func(dst unsafe.Pointer, src unsafe.Pointer, words int) {
		copy(unsafe.Slice((*uint64)(dst), words), unsafe.Slice((*uint64)(src), words))
	}
	copyPt(unsafe.Pointer(&pk.G1.Alpha), unsafe.Pointer(&out.g1_alpha[0]), 8)
	copyPt(unsafe.Pointer(&pk.G1.Beta), unsafe.Pointer(&out.g1_beta[0]), 8)
	copyPt(unsafe.Pointer(&pk.G1.Delta), unsafe.Pointer(&out.g1_delta[0]), 8)
	copyPt(unsafe.Pointer(&pk.G2.Beta), unsafe.Pointer(&out.g2_beta[0]), 16)
	copyPt(unsafe.Pointer(&pk.G2.Delta), unsafe.Pointer(&out.g2_delta[0]), 16)

	vk := &groth16_bn254.VerifyingKey{}
	vk.G1.Alpha, vk.G1.Beta, vk.G1.Delta = pk.G1.Alpha, pk.G1.Beta, pk.G1.Delta
	vk.G2.Beta, vk.G2.Delta = pk.G2.Beta, pk.G2.Delta
	copyPt(unsafe.Pointer(&vk.G2.Gamma), unsafe.Pointer(&out.g2_gamma[0]), 16)
	if vk.G1.K, err = g1(out.vk_k); err != nil {
		return fail(err)
	}
	if len(commitmentInfo) == 1 {
		var ck pedersen.ProvingKey
		if ck.Basis, err = g1(out.ped_basis); err == nil {
			ck.BasisExpSigma, err = g1(out.ped_basis_exp_sigma)
		}
		if err != nil {
			return fail(err)
		}
		pk.CommitmentKeys = []pedersen.ProvingKey{ck}
		var vck pedersen.VerifyingKey
		copyPt(unsafe.Pointer(&vck.G), unsafe.Pointer(&out.ped_g[0]), 16)
		copyPt(unsafe.Pointer(&vck.GSigmaNeg), unsafe.Pointer(&out.ped_g_sigma_neg[0]), 16)
		vk.CommitmentKeys = []pedersen.VerifyingKey{vck}
		vk.PublicAndCommitmentCommitted = [][]int{publicCommitted}
	}
	if err := vk.Precompute(); err != nil {
		return fail(err)
	}

	// the resident vectors become the device key (borrowed by the pk handle, released with it by Free)
	dd := C.b200g16_pk_desc{
		log2_domain: out.log2_domain, n_wires: C.size_t(nbWires),
		res_a: out.a, res_b: out.b, res_k: out.k, res_z: out.z, res_b2: out.b2,
		n_a: C.size_t(len(pk.G1.A)), n_b: C.size_t(len(pk.G1.B)), n_k: C.size_t(len(pk.G1.K)), n_z: C.size_t(len(pk.G1.Z)),
		g1_alpha: &out.g1_alpha[0], g1_beta: &out.g1_beta[0], g1_delta: &out.g1_delta[0],
		g2_beta: &out.g2_beta[0], g2_delta: &out.g2_delta[0],
		infinity_a: (*C.uint8_t)(unsafe.Pointer(&infA[0])), infinity_b: (*C.uint8_t)(unsafe.Pointer(&infB[0])),
		k_skip: (*C.uint8_t)(unsafe.Pointer(&kSkip[0])),
	}
	if err := call(func() C.int { return C.b200g16_pk_upload(pk.ctx, &dd, &pk.dev) }); err != nil {
		return fail(err)
	}
	return pk, vk, nil
}
