// One Go process, several GPUs: gnark calls groth16.Prove once (mt.go:496); a group spreads that one call over the
// GPUs of the box through libb200g16's b200g16_group_* entry points (no NCCL, no helper processes).
// NOT built or tested in this repository (no Go toolchain); the same calls run in tests/test_gpu_group.py via ctypes.
//go:build b200

package b200

/*
#include "b200g16.h"
*/
import "C"

import (
	"errors"
	"math/bits"
	"runtime"
	"unsafe"

	curve "github.com/consensys/gnark-crypto/ecc/bn254"
	"github.com/consensys/gnark-crypto/ecc/bn254/fr"
	groth16_bn254 "github.com/consensys/gnark/backend/groth16/bn254"
	cs "github.com/consensys/gnark/constraint/bn254"
)

// GroupProvingKey = gnark's pk + its point-range shards resident on every GPU of the group.
type GroupProvingKey struct {
	groth16_bn254.ProvingKey
	grp *C.b200g16_group
	dev *C.b200g16_group_pk
}

// Upload cuts the key into one shard per device (devices = CUDA ordinals) and builds the window tables there.
func (pk *GroupProvingKey) Upload(devices []int, kSkip []byte) error {
	devs := make([]C.int, len(devices))
	for i, d := range devices {
		devs[i] = C.int(d)
	}
	if err := call(func() C.int { return C.b200g16_group_init(&devs[0], C.int(len(devs)), &pk.grp) }); err != nil {
		return err
	}
	infA, infB := boolsToBytes(pk.InfinityA), boolsToBytes(pk.InfinityB)
	var pin runtime.Pinner
	defer pin.Unpin()
	for _, p := range []any{&pk.G1.A[0], &pk.G1.B[0], &pk.G1.K[0], &pk.G1.Z[0], &pk.G2.B[0], &pk.G1.Alpha, &pk.G1.Beta,
		&pk.G1.Delta, &pk.G2.Beta, &pk.G2.Delta, &infA[0], &infB[0], &kSkip[0]} {
		pin.Pin(p)
	}
	d := C.b200g16_pk_desc{
		log2_domain: C.uint(bits.TrailingZeros64(pk.Domain.Cardinality)),
		n_wires:     C.size_t(len(pk.InfinityA)),
		g1_a:        u64(unsafe.Pointer(&pk.G1.A[0])), n_a: C.size_t(len(pk.G1.A)),
		g1_b:        u64(unsafe.Pointer(&pk.G1.B[0])), n_b: C.size_t(len(pk.G1.B)),
		g1_k:        u64(unsafe.Pointer(&pk.G1.K[0])), n_k: C.size_t(len(pk.G1.K)),
		g1_z:        u64(unsafe.Pointer(&pk.G1.Z[0])), n_z: C.size_t(len(pk.G1.Z)),
		g2_b:        u64(unsafe.Pointer(&pk.G2.B[0])),
		g1_alpha:    u64(unsafe.Pointer(&pk.G1.Alpha)), g1_beta: u64(unsafe.Pointer(&pk.G1.Beta)),
		g1_delta:    u64(unsafe.Pointer(&pk.G1.Delta)),
		g2_beta:     u64(unsafe.Pointer(&pk.G2.Beta)), g2_delta: u64(unsafe.Pointer(&pk.G2.Delta)),
		infinity_a:  (*C.uint8_t)(unsafe.Pointer(&infA[0])), infinity_b: (*C.uint8_t)(unsafe.Pointer(&infB[0])),
		k_skip:      (*C.uint8_t)(unsafe.Pointer(&kSkip[0])),
		precompute:  1,
	}
	return call(func() C.int { return C.b200g16_group_pk_upload(pk.grp, &d, &pk.dev) })
}

// ProveSolved runs everything after the constraint solver on all GPUs of the group: computeH split over the
// devices (2, 4 or 8: cross-GPU NTT levels over NVLink peer memory), the five MSMs on every shard, the partial
// points added on the host.  r, s as in b200.Prove.
func (pk *GroupProvingKey) ProveSolved(solution *cs.R1CSSolution, r, s *fr.Element) (*groth16_bn254.Proof, error) {
	wires := []fr.Element(solution.W)
	var out C.b200g16_proof
	err := call(func() C.int {
		return C.b200g16_group_prove(pk.grp, pk.dev,
			u64(unsafe.Pointer(&wires[0])), C.size_t(len(wires)),
			u64(unsafe.Pointer(&solution.A[0])), u64(unsafe.Pointer(&solution.B[0])), u64(unsafe.Pointer(&solution.C[0])),
			C.size_t(len(solution.A)), u64(unsafe.Pointer(r)), u64(unsafe.Pointer(s)), &out, nil)
	})
	if err != nil {
		return nil, err
	}
	proof := &groth16_bn254.Proof{}
	proof.Ar = *(*curve.G1Affine)(unsafe.Pointer(&out.ar))
	proof.Bs = *(*curve.G2Affine)(unsafe.Pointer(&out.bs))
	proof.Krs = *(*curve.G1Affine)(unsafe.Pointer(&out.krs))
	return proof, nil
}

func (pk *GroupProvingKey) Free() {
	if pk.dev != nil {
		C.b200g16_group_pk_free(pk.dev)
		pk.dev = nil
	}
	if pk.grp != nil {
		C.b200g16_group_destroy(pk.grp)
		pk.grp = nil
	}
}

// ReplicatedKey = a whole resident single-GPU key on every GPU of a group, for throughput: each device proves whole
// proofs of its own share of a batch, with no data crossing devices.
type ReplicatedKey struct {
	grp *C.b200g16_group
	dev *C.b200g16_group_pk
}

// Replicate starts a group over devices (CUDA ordinals) and makes pk's resident key (from Setup, or uploaded by a
// first Prove / BatchProve) available on every one of them: devices other than pk's receive device-to-device
// copies of the point vectors, window tables included.  pk must outlive the replicated key.
func Replicate(pk *ProvingKey, devices []int) (*ReplicatedKey, error) {
	if pk.dev == nil {
		return nil, errors.New("b200: Replicate needs a resident key (Setup, or one Prove / BatchProve first)")
	}
	if len(devices) == 0 {
		return nil, errors.New("b200: Replicate needs at least one device")
	}
	devs := make([]C.int, len(devices))
	for i, d := range devices {
		devs[i] = C.int(d)
	}
	rk := &ReplicatedKey{}
	if err := call(func() C.int { return C.b200g16_group_init(&devs[0], C.int(len(devs)), &rk.grp) }); err != nil {
		return nil, err
	}
	if err := call(func() C.int { return C.b200g16_group_pk_replicate(rk.grp, pk.dev, &rk.dev) }); err != nil {
		rk.Free()
		return nil, err
	}
	return rk, nil
}

// BatchProveSolved proves k solved witnesses of one circuit over the group, rs[j], ss[j] the blinding scalars of
// proof j: one b200g16_group_prove_batch call, the proofs split into contiguous ranges over the devices.  Proof j
// equals BatchProve's proof for the same solution and r, s.  A circuit's commitments and proofs of knowledge are the
// caller's, as in ProveSolved.
func (rk *ReplicatedKey) BatchProveSolved(solutions []*cs.R1CSSolution, rs, ss []fr.Element) ([]*groth16_bn254.Proof, error) {
	k := len(solutions)
	if len(rs) != k || len(ss) != k {
		return nil, errors.New("b200: BatchProveSolved needs one r and one s per solution")
	}
	if k == 0 {
		return nil, nil
	}
	nWires, nCons := len(solutions[0].W), len(solutions[0].A)
	wires := make([]fr.Element, 0, k*nWires)
	A := make([]fr.Element, 0, k*nCons)
	B := make([]fr.Element, 0, k*nCons)
	Cv := make([]fr.Element, 0, k*nCons)
	for _, sol := range solutions {
		if len(sol.W) != nWires || len(sol.A) != nCons || len(sol.B) != nCons || len(sol.C) != nCons {
			return nil, errors.New("b200: BatchProveSolved needs solutions of one circuit")
		}
		wires = append(wires, sol.W...)
		A = append(A, sol.A...)
		B = append(B, sol.B...)
		Cv = append(Cv, sol.C...)
	}
	out := make([]C.b200g16_proof, k)
	err := call(func() C.int {
		return C.b200g16_group_prove_batch(rk.grp, rk.dev, C.size_t(k), u64(unsafe.Pointer(&wires[0])), C.size_t(nWires),
			u64(unsafe.Pointer(&A[0])), u64(unsafe.Pointer(&B[0])), u64(unsafe.Pointer(&Cv[0])), C.size_t(nCons),
			u64(unsafe.Pointer(&rs[0])), u64(unsafe.Pointer(&ss[0])), &out[0])
	})
	if err != nil {
		return nil, err
	}
	proofs := make([]*groth16_bn254.Proof, k)
	for j := range proofs {
		proofs[j] = &groth16_bn254.Proof{}
		proofs[j].Ar = *(*curve.G1Affine)(unsafe.Pointer(&out[j].ar))
		proofs[j].Bs = *(*curve.G2Affine)(unsafe.Pointer(&out[j].bs))
		proofs[j].Krs = *(*curve.G1Affine)(unsafe.Pointer(&out[j].krs))
	}
	return proofs, nil
}

// Free releases the copies and the group (never the source key).
func (rk *ReplicatedKey) Free() {
	if rk.dev != nil {
		C.b200g16_group_pk_free(rk.dev)
		rk.dev = nil
	}
	if rk.grp != nil {
		C.b200g16_group_destroy(rk.grp)
		rk.grp = nil
	}
}
