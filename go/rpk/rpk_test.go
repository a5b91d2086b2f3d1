package rpk

// Tests a maintainer runs after dropping the engine under pkg/virtual_kubelet (needs a B200 and the built
// librpk.so; see the build line in rpk.go).  NOT EXECUTED in this repository: the image has no Go toolchain
// (SURVEY.md 8c).  The same scenarios run here through the same C-ABI from C++ (host/host_test.cc) and Python
// (tests/test_select_gpu.py::test_kat_table, tests/test_oracle.py::test_column_producers_golden).
//
// Scenario sources: the column-producer cases are the assertions of the reference's own tests
// (annotations_test.go:117-118, 141-142, 233-234, 121-122, 225-226; runpod_test.go:89-90); the selection cases
// are the known answers derived in SURVEY.md 8(c) from runpod_client.go:465-509 (the reference has no test that
// pins gpuTypeIds).

import (
	"reflect"
	"testing"
)

// The ten-offer table of SURVEY.md 8(c); index = position = offer id.
func katOffers() *Offers {
	type row struct {
		id       string
		mem      int32
		sec      bool
		secPrice float64
		com      bool
		comPrice float64
	}
	rows := []row{
		{"A4000", 16, true, 0.32, true, 0.17},
		{"A5000", 24, true, 0.36, true, 0.22},
		{"RTX3090", 24, false, 0, true, 0.22},
		{"A40", 48, true, 0.40, false, 0},
		{"RTX4090", 24, true, 0.69, true, 0.34},
		{"L4", 24, true, 0.43, false, 0},
		{"A100", 80, true, 1.64, true, 1.19},
		{"T4free", 16, true, 0, true, 0},
		{"A4500", 20, true, 0.34, true, 0.19},
		{"edge", 32, true, 0.5, true, 0.5},
	}
	o := &Offers{}
	for _, r := range rows {
		o.IDs = append(o.IDs, r.id)
		o.MemoryInGb = append(o.MemoryInGb, r.mem)
		o.SecurePrice = append(o.SecurePrice, r.secPrice)
		o.CommunityPrice = append(o.CommunityPrice, r.comPrice)
		var f uint8
		if r.sec {
			f |= 1
		}
		if r.com {
			f |= 2
		}
		o.Flags = append(o.Flags, f)
	}
	return o
}

func trim(top5 []int32) []int32 {
	out := []int32{}
	for _, v := range top5 {
		if v >= 0 {
			out = append(out, v)
		}
	}
	return out
}

// GetGPUTypes(minRAMPerGPU, maxPrice, cloudType) for one pod at a time, as the reference calls it
// (runpod_client.go:1281), and for all cases as one batch: both must give the same lists.
func TestSelectKnownAnswers(t *testing.T) {
	e, err := New(1)
	if err != nil {
		t.Skipf("no B200: %v", err)
	}
	defer e.Close()
	if err := e.UploadOffers(katOffers()); err != nil {
		t.Fatal(err)
	}
	cases := []struct {
		name     string
		minMem   int32
		maxPrice float64
		cloud    uint8
		want     []int32
	}{
		{"ordering, price 0 excluded, strict < 0.5", 16, 0.5, CloudSecure, []int32{0, 8, 1, 3, 5}},
		{"mem >= min", 24, 0.5, CloudSecure, []int32{1, 3, 5}},
		{"tie 0.22 -> lower index first", 24, 0.5, CloudCommunity, []int32{1, 2, 4}},
		{"single", 48, 0.5, CloudSecure, []int32{3}},
		{"empty is not an error", 80, 0.5, CloudSecure, []int32{}},
		{"neither SECURE nor COMMUNITY", 16, 0.5, 7, []int32{}},
		{"exactly five", 2, 0.5, CloudCommunity, []int32{0, 8, 1, 2, 4}},
		{"eight feasible truncated to five", 16, 2.0, CloudSecure, []int32{0, 8, 1, 3, 5}},
	}
	batch := &Pods{}
	for _, c := range cases {
		one := &Pods{ReqMemGb: []int32{c.minMem}, MaxPrice: []float64{c.maxPrice}, Cloud: []uint8{c.cloud}}
		best, top5, err := e.Select(one, true)
		if err != nil {
			t.Fatalf("%s: %v", c.name, err)
		}
		if got := trim(top5); !reflect.DeepEqual(got, c.want) {
			t.Errorf("%s: gpuTypeIds = %v, want %v", c.name, got, c.want)
		}
		wantBest := int32(-1)
		if len(c.want) > 0 {
			wantBest = c.want[0]
		}
		if best[0] != wantBest {
			t.Errorf("%s: best = %d, want %d", c.name, best[0], wantBest)
		}
		batch.ReqMemGb = append(batch.ReqMemGb, c.minMem)
		batch.MaxPrice = append(batch.MaxPrice, c.maxPrice)
		batch.Cloud = append(batch.Cloud, c.cloud)
	}
	_, top5, err := e.Select(batch, true)
	if err != nil {
		t.Fatal(err)
	}
	for i, c := range cases {
		if got := trim(top5[i*TopK : (i+1)*TopK]); !reflect.DeepEqual(got, c.want) {
			t.Errorf("batched %s: gpuTypeIds = %v, want %v", c.name, got, c.want)
		}
	}
}

// The assertions of annotations_test.go / runpod_test.go on the (minRAMPerGPU, cloudType) pair.
func TestColumnProducers(t *testing.T) {
	const memKey, cloudKey = "runpod.io/required-gpu-memory", "runpod.io/cloud-type"
	cases := []struct {
		name      string
		pod, job  map[string]string
		wantMem   int32
		wantCloud uint8
	}{
		{"job annotation only (annotations_test.go:117,121)", map[string]string{}, map[string]string{memKey: "8", cloudKey: "SECURE"}, 8, CloudSecure},
		{"pod overrides job (annotations_test.go:141)", map[string]string{memKey: "16"}, map[string]string{memKey: "8"}, 16, CloudSecure},
		{"job fallback, pod cloud wins (annotations_test.go:225,233)", map[string]string{cloudKey: "SECURE"}, map[string]string{memKey: "24", cloudKey: "COMMUNITY"}, 24, CloudSecure},
		{"STANDARD falls to SECURE (runpod_test.go:89-90)", map[string]string{memKey: "2", cloudKey: "STANDARD"}, nil, 2, CloudSecure},
		{"defaults", map[string]string{}, nil, 16, CloudSecure},
		{"parse error -> 16", map[string]string{memKey: "lots"}, nil, 16, CloudSecure},
		{"lower case community", map[string]string{cloudKey: "community"}, nil, 16, CloudCommunity},
		{"huge request saturates", map[string]string{memKey: "99999999999"}, nil, 1<<31 - 1, CloudSecure},
	}
	for _, c := range cases {
		if got := ReqMemColumn(AnnotationWithFallback(c.pod, c.job, memKey, "")); got != c.wantMem {
			t.Errorf("%s: minRAMPerGPU = %d, want %d", c.name, got, c.wantMem)
		}
		if got := CloudColumn(AnnotationWithFallback(c.pod, c.job, cloudKey, "")); got != c.wantCloud {
			t.Errorf("%s: cloud = %d, want %d", c.name, got, c.wantCloud)
		}
	}
}

// kubelet.go:870-873: a slot reports iff its (status, ports) pair changed since the previous sweep.
func TestStatusDiff(t *testing.T) {
	e, err := New(1)
	if err != nil {
		t.Skipf("no B200: %v", err)
	}
	defer e.Close()
	const stride = 32
	states := []struct {
		status string
		ports  bool
	}{{"STARTING", false}, {"RUNNING", false}, {"RUNNING", true}, {"EXITED", true}}
	recs := make([]byte, len(states)*stride)
	for i, s := range states {
		if err := EncodeStatusRecord(recs[i*stride:(i+1)*stride], s.status, s.ports, false); err != nil {
			t.Fatal(err)
		}
	}
	if err := e.StatusSeed(recs, stride); err != nil { // CreatePod / LoadRunning wrote InstanceInfo
		t.Fatal(err)
	}
	if got, err := e.StatusDiff(recs, stride); err != nil || len(got) != 0 {
		t.Fatalf("unchanged sweep reported %v (err %v)", got, err)
	}
	_ = EncodeStatusRecord(recs[0*stride:1*stride], "RUNNING", false, false) // status changed
	_ = EncodeStatusRecord(recs[1*stride:2*stride], "RUNNING", true, false)  // only the ports bit changed
	got, err := e.StatusDiff(recs, stride)
	if err != nil {
		t.Fatal(err)
	}
	if want := []uint32{0, 1}; !reflect.DeepEqual(got, want) {
		t.Errorf("changed = %v, want %v", got, want)
	}
}

// runpod.io/gpu-type-ids: parsed like runpod.io/datacenter-ids (runpod_client.go:1354-1362).
func TestGpuTypeIDs(t *testing.T) {
	cases := []struct {
		in   string
		want []string
	}{
		{"", nil},
		{"A40", []string{"A40"}},
		{" A40 , L4\t,A100 ", []string{"A40", "L4", "A100"}},
		{"A40,,L4", []string{"A40", "", "L4"}},
		{",", []string{"", ""}},
	}
	for _, c := range cases {
		if got := GpuTypeIDs(c.in); !reflect.DeepEqual(got, c.want) {
			t.Errorf("GpuTypeIDs(%q) = %q, want %q", c.in, got, c.want)
		}
	}
}

// The offer-set known answers of tests/golden/select_sets_kat.json: a restricted pod gets GetGPUTypes over its
// set's members only, table indices out, ties to the lower table index whatever the list order.
func TestSelectSetsKnownAnswers(t *testing.T) {
	e, err := New(1)
	if err != nil {
		t.Skipf("no B200: %v", err)
	}
	defer e.Close()
	if err := e.UploadOffers(katOffers()); err != nil {
		t.Fatal(err)
	}
	sets := [][]int32{{1, 3, 5}, {2}, {4, 2, 1}, {6, 7, 9}, {}} // {A5000, A40, L4}, {RTX3090}, ..., ids not in the table
	if err := e.UploadOfferSets(sets); err != nil {
		t.Fatal(err)
	}
	cases := []struct {
		name     string
		minMem   int32
		maxPrice float64
		cloud    uint8
		set      uint16
		want     []int32
	}{
		{"price order inside the set", 16, 0.5, CloudSecure, 0, []int32{1, 3, 5}},
		{"only member has no secure flag", 16, 0.5, CloudSecure, 1, []int32{}},
		{"tie 0.22 -> lower table index", 24, 0.5, CloudCommunity, 2, []int32{1, 2, 4}},
		{"price 0 excluded; 0.5 < 2.0", 16, 2.0, CloudSecure, 3, []int32{9, 6}},
		{"empty set", 16, 0.5, CloudSecure, 4, []int32{}},
		{"id without a set", 16, 0.5, CloudSecure, 17, []int32{}},
		{"unrestricted = the reference KAT", 16, 0.5, CloudSecure, SetAll, []int32{0, 8, 1, 3, 5}},
	}
	batch := &Pods{}
	var ids []uint16
	for _, c := range cases {
		batch.ReqMemGb = append(batch.ReqMemGb, c.minMem)
		batch.MaxPrice = append(batch.MaxPrice, c.maxPrice)
		batch.Cloud = append(batch.Cloud, c.cloud)
		ids = append(ids, c.set)
	}
	best, top5, err := e.SelectSets(batch, ids, true)
	if err != nil {
		t.Fatal(err)
	}
	for i, c := range cases {
		if got := trim(top5[i*TopK : (i+1)*TopK]); !reflect.DeepEqual(got, c.want) {
			t.Errorf("%s: gpuTypeIds = %v, want %v", c.name, got, c.want)
		}
		wantBest := int32(-1)
		if len(c.want) > 0 {
			wantBest = c.want[0]
		}
		if best[i] != wantBest {
			t.Errorf("%s: best = %d, want %d", c.name, best[i], wantBest)
		}
	}
	if err := e.UploadOffers(katOffers()); err != nil { // a new table makes the sets stale
		t.Fatal(err)
	}
	if _, _, err := e.SelectSets(batch, ids, false); err == nil {
		t.Errorf("SelectSets after UploadOffers: want an error (stale offer sets)")
	}
}
