// Source a maintainer adds to gnark-whir (or to a gnark fork) to put libb200g16 behind gnark's groth16 API.
// NOT built or tested in this repository: the image has no Go toolchain (see INTEGRATION.md).  The same C-ABI,
// call for call, is exercised by gnark_whir_b200/lib.py + groth16.py in the test-suite.
//go:build b200

package b200

/*
#include "b200g16.h"
*/
import "C"

import (
	"crypto/rand"
	"errors"
	"fmt"
	"unsafe"

	"github.com/consensys/gnark-crypto/ecc/bn254/fr"
	"github.com/consensys/gnark-crypto/ecc/bn254/fr/hash_to_field"
	groth16_bn254 "github.com/consensys/gnark/backend/groth16/bn254"
	"github.com/consensys/gnark/constraint"
)

// publicInputs: the public inputs b200g16_verify takes for one proof — the public witness, then, when the circuit
// has a BSB22 commitment, the challenge hash_to_field("bsb22-commitment")(proof.Commitments[0].Marshal() ||
// committed publics), exactly as gnark v0.11.0 verify.go computes it
func publicInputs(proof *groth16_bn254.Proof, vk *groth16_bn254.VerifyingKey, publicWitness fr.Vector) fr.Vector {
	pub := append(fr.Vector{}, publicWitness...)
	if len(vk.PublicAndCommitmentCommitted) > 0 { // one BSB22 commitment (what this circuit has)
		h := hash_to_field.New([]byte(constraint.CommitmentDst))
		maxNb := len(vk.PublicAndCommitmentCommitted[0])
		buf := make([]byte, 0, 64+maxNb*fr.Bytes)
		buf = append(buf, proof.Commitments[0].Marshal()...)
		for _, w := range vk.PublicAndCommitmentCommitted[0] {
			b := pub[w-1].Bytes() // wire ids count the constant-one wire; publicWitness does not hold it
			buf = append(buf, b[:]...)
		}
		h.Write(buf)
		var challenge fr.Element
		challenge.SetBytes(h.Sum(nil)[:fr.Bytes])
		pub = append(pub, challenge)
	}
	return pub
}

func vkDesc(vk *groth16_bn254.VerifyingKey) C.b200g16_vk_desc {
	d := C.b200g16_vk_desc{
		g1_alpha: u64(unsafe.Pointer(&vk.G1.Alpha)), g2_beta: u64(unsafe.Pointer(&vk.G2.Beta)),
		g2_gamma: u64(unsafe.Pointer(&vk.G2.Gamma)), g2_delta: u64(unsafe.Pointer(&vk.G2.Delta)),
		g1_k: u64(unsafe.Pointer(&vk.G1.K[0])), n_k: C.size_t(len(vk.G1.K)),
	}
	if len(vk.PublicAndCommitmentCommitted) > 0 {
		d.ped_g = u64(unsafe.Pointer(&vk.CommitmentKeys[0].G))
		d.ped_g_sigma_neg = u64(unsafe.Pointer(&vk.CommitmentKeys[0].GSigmaNeg))
	}
	return d
}

// groth16.Verify(proof, vk, publicWitness) at mt.go:497
func Verify(ctx *C.b200g16_ctx, proof *groth16_bn254.Proof, vk *groth16_bn254.VerifyingKey, publicWitness fr.Vector) error {
	pub := publicInputs(proof, vk, publicWitness)
	var com, pok *C.uint64_t
	if len(vk.PublicAndCommitmentCommitted) > 0 {
		com, pok = u64(unsafe.Pointer(&proof.Commitments[0])), u64(unsafe.Pointer(&proof.CommitmentPok))
	}
	d := vkDesc(vk)
	var ok C.int
	if err := call(func() C.int {
		return C.b200g16_verify(ctx, &d, u64(unsafe.Pointer(&proof.Ar)), u64(unsafe.Pointer(&proof.Bs)),
			u64(unsafe.Pointer(&proof.Krs)), com, pok, u64(unsafe.Pointer(&pub[0])), C.size_t(len(pub)), &ok)
	}); err != nil {
		return err                                           // malformed input ("invalid witness size", bad point)
	}
	if ok == 0 { return errors.New("pairing doesn't match") } // gnark's errPairingCheckFailed
	return nil
}

// BatchVerify checks len(proofs) proofs of one circuit in one b200g16_verify_batch call and returns, per proof, what
// Verify would decide for it alone.  The batch coefficients come from crypto/rand after the proofs are fixed: the
// test is sound (a bad batch passes with probability about 2^-128) only while whoever made the proofs cannot predict
// them.  An error means malformed input, as from Verify.
func BatchVerify(ctx *C.b200g16_ctx, proofs []*groth16_bn254.Proof, vk *groth16_bn254.VerifyingKey, publicWitnesses []fr.Vector) ([]bool, error) {
	k := len(proofs)
	if len(publicWitnesses) != k {
		return nil, fmt.Errorf("%d proofs but %d public witnesses", k, len(publicWitnesses))
	}
	if k == 0 {
		return []bool{}, nil
	}
	hasCom := len(vk.PublicAndCommitmentCommitted) > 0
	nPub := len(vk.G1.K) - 1
	// Go-allocated, pointer-free buffers: cgo may pass them for the duration of the call
	ar := make([]uint64, 8*k)
	bs := make([]uint64, 16*k)
	krs := make([]uint64, 8*k)
	pub := make([]uint64, 4*nPub*k+1)
	var com, pok []uint64
	if hasCom {
		com, pok = make([]uint64, 8*k), make([]uint64, 8*k)
	}
	for i, p := range proofs {
		x := publicInputs(p, vk, publicWitnesses[i])
		if len(x) != nPub {
			return nil, fmt.Errorf("proof %d: invalid witness size %d, vk.G1.K expects %d", i, len(x), nPub)
		}
		copy(ar[8*i:], (*[8]uint64)(unsafe.Pointer(&p.Ar))[:])
		copy(bs[16*i:], (*[16]uint64)(unsafe.Pointer(&p.Bs))[:])
		copy(krs[8*i:], (*[8]uint64)(unsafe.Pointer(&p.Krs))[:])
		for j := range x {
			copy(pub[4*(nPub*i+j):], x[j][:])
		}
		if hasCom {
			if len(p.Commitments) == 0 {
				return nil, fmt.Errorf("proof %d carries no commitment but the circuit has one", i)
			}
			copy(com[8*i:], (*[8]uint64)(unsafe.Pointer(&p.Commitments[0]))[:])
			copy(pok[8*i:], (*[8]uint64)(unsafe.Pointer(&p.CommitmentPok))[:])
		}
	}
	nCoef := k
	if hasCom {
		nCoef = 2 * k
	}
	coeffs := make([]uint64, 2*nCoef)
	buf := make([]byte, 16)
	for i := 0; i < nCoef; i++ {
		for coeffs[2*i] == 0 && coeffs[2*i+1] == 0 { // redraw the (2^-128) zero
			if _, err := rand.Read(buf); err != nil {
				return nil, err
			}
			for b := 0; b < 8; b++ {
				coeffs[2*i] |= uint64(buf[b]) << (8 * b)
				coeffs[2*i+1] |= uint64(buf[8+b]) << (8 * b)
			}
		}
	}
	var comP, pokP *C.uint64_t
	if hasCom {
		comP, pokP = u64(unsafe.Pointer(&com[0])), u64(unsafe.Pointer(&pok[0]))
	}
	d := vkDesc(vk)
	var ok C.int
	each := make([]byte, k)
	if err := call(func() C.int {
		return C.b200g16_verify_batch(ctx, &d, C.size_t(k), u64(unsafe.Pointer(&ar[0])), u64(unsafe.Pointer(&bs[0])),
			u64(unsafe.Pointer(&krs[0])), comP, pokP, u64(unsafe.Pointer(&pub[0])), C.size_t(nPub),
			u64(unsafe.Pointer(&coeffs[0])), &ok, (*C.uint8_t)(unsafe.Pointer(&each[0])))
	}); err != nil {
		return nil, err
	}
	res := make([]bool, k)
	for i := range res {
		res[i] = each[i] != 0
	}
	return res, nil
}
