package muse

/*
#cgo CFLAGS: -I${SRCDIR}/../../../include
#cgo LDFLAGS: -L${SRCDIR}/../.. -lmuse_b200
#include <stdlib.h>
#include "muse_b200.h"
*/
import "C"

import (
	"errors"
	"fmt"
	"os"
	"runtime"
	"sort"
	"strconv"
	"sync"
	"unsafe"
)

var (
	ctxOnce sync.Once
	ctx     *C.muse_ctx
	ctxErr  error
)

func lastError(rc C.int) error {
	return fmt.Errorf("muse_b200: %s (status %d)", C.GoString(C.muse_last_error()), int(rc))
}

// deviceContext creates the process-wide context on device MUSE_DEVICE (default 0; one process per GPU sets it to its
// local rank).
func deviceContext() (*C.muse_ctx, error) {
	ctxOnce.Do(func() {
		dev := 0
		if v := os.Getenv("MUSE_DEVICE"); v != "" {
			d, err := strconv.Atoi(v)
			if err != nil || d < 0 {
				ctxErr = fmt.Errorf("muse_b200: MUSE_DEVICE=%q is not a device index", v)
				return
			}
			dev = d
		}
		if rc := C.muse_ctx_create(C.int(dev), &ctx); rc != C.MUSE_OK {
			ctxErr = lastError(rc)
		}
	})
	return ctx, ctxErr
}

// Group is a collection of uniquely labelled timeseries of one length (go-muse group.go:7-104).
// The values live in a device-resident fp64 slab; label values are dictionary encoded to int32
// ids per key (strings never cross the C boundary).
type Group struct {
	Name     string
	n        int
	registry map[string]int // uid -> index into series
	series   []*Series

	store    *C.muse_group
	gen      uint64                    // bumped whenever the device store is replaced: a Batch bound to an older one rebinds
	cols     []string                  // label key of each device column (the last column is all -1)
	dict     map[string]map[string]int32
	uploaded int

	// sharded groups (exchange.go): index of this block's first series in the whole group, and the label dictionary
	// every process agreed on
	shardFirst int64
	fixedDict  map[string][]string
}

// uploadChunk is the number of series handed to muse_group_append per call: the library copies the rows (through its
// pinned staging ring when they sit in pageable Go memory), so nothing larger than one chunk is ever duplicated on the host.
const uploadChunk = 4096

// NewGroup creates a new Group and initializes the timeseries label registry.
func NewGroup(name string) *Group {
	g := &Group{Name: name, registry: make(map[string]int)}
	runtime.SetFinalizer(g, func(g *Group) {
		if g.store != nil {
			C.muse_group_destroy(g.store)
		}
	})
	return g
}

// Length returns the length of all timeseries.
func (g *Group) Length() int { return g.n }

// Add registers time series; errors mirror go-muse group.go:31-56.
func (g *Group) Add(series ...*Series) error {
	for _, s := range series {
		if len(s.lab.Keys()) == 0 {
			return fmt.Errorf("Invalid Series with no labels, %v", s)
		}
		uid := s.UID()
		if _, exists := g.registry[uid]; exists {
			return fmt.Errorf("Series with label:values, %v, already exists within group, %s", uid, g.Name)
		}
		if len(g.registry) == 0 {
			g.n = s.Length()
		} else if s.Length() != g.n {
			return fmt.Errorf("Timeseries has length %d, but current group has length %d", s.Length(), g.n)
		}
		g.registry[uid] = len(g.series)
		g.series = append(g.series, s)
	}
	return nil
}

// FilterByLabelValues returns the series whose values match on every key of labels.
func (g *Group) FilterByLabelValues(labels *Labels) []*Series {
	keys := labels.Keys()
	if len(keys) == 0 {
		return nil
	}
	want := labels.ID(append([]string(nil), keys...))
	var out []*Series
	for _, s := range g.series {
		if s.lab.ID(append([]string(nil), keys...)) == want {
			out = append(out, s)
		}
	}
	return out
}

// syncDevice uploads series added since the last call (muse_group_append copies the rows, so no
// Go pointer is retained by C).
func (g *Group) syncDevice() error {
	c, err := deviceContext()
	if err != nil {
		return err
	}
	keySet := map[string]struct{}{}
	for k := range g.fixedDict { // sharded: every process has the same columns, whatever its own series carry
		keySet[k] = struct{}{}
	}
	for _, s := range g.series {
		for _, k := range s.lab.Keys() {
			keySet[k] = struct{}{}
		}
	}
	keys := make([]string, 0, len(keySet))
	for k := range keySet {
		keys = append(keys, k)
	}
	sort.Strings(keys)
	same := len(keys) == len(g.cols)
	for i := 0; same && i < len(keys); i++ {
		same = keys[i] == g.cols[i]
	}
	if g.store == nil || !same {
		if g.store != nil {
			C.muse_group_destroy(g.store)
			g.store = nil
		}
		g.gen++
		g.cols = keys
		g.dict = make(map[string]map[string]int32)
		for _, k := range keys {
			g.dict[k] = make(map[string]int32)
			for i, v := range g.fixedDict[k] {
				g.dict[k][v] = int32(i)
			}
		}
		if rc := C.muse_group_create(c, C.int64_t(g.n), C.int32_t(len(keys)+1), C.int64_t(len(g.series)), &g.store); rc != C.MUSE_OK {
			return lastError(rc)
		}
		if g.shardFirst != 0 {
			if rc := C.muse_group_set_global_offset(g.store, C.int64_t(g.shardFirst)); rc != C.MUSE_OK {
				return lastError(rc)
			}
		}
		g.uploaded = 0
	}
	if g.uploaded == len(g.series) {
		return nil
	}
	nk := len(g.cols) + 1
	rows := make([]float64, 0, uploadChunk*g.n)
	ids := make([]int32, 0, uploadChunk*nk)
	for g.uploaded < len(g.series) {
		end := g.uploaded + uploadChunk
		if end > len(g.series) {
			end = len(g.series)
		}
		rows, ids = rows[:0], ids[:0]
		for _, s := range g.series[g.uploaded:end] {
			rows = append(rows, s.vals...)
			base := len(ids)
			for c := 0; c < nk; c++ {
				ids = append(ids, -1)
			}
			for c, k := range g.cols {
				if v, ok := s.lab.Get(k); ok {
					d := g.dict[k]
					id, seen := d[v]
					if !seen {
						id = int32(len(d))
						d[v] = id
					}
					ids[base+c] = id
				}
			}
		}
		rc := C.muse_group_append(g.store, (*C.double)(unsafe.Pointer(&rows[0])), C.int64_t(end-g.uploaded), C.int64_t(g.n),
			(*C.int32_t)(unsafe.Pointer(&ids[0])))
		if rc != C.MUSE_OK {
			return lastError(rc)
		}
		g.uploaded = end
	}
	return nil
}

// rollChunkBytes bounds the new samples handed to muse_group_roll per call: the library copies them (through its pinned
// staging ring when they sit in pageable Go memory), so nothing larger than one chunk is duplicated on the host.
const rollChunkBytes = 64 << 20

// Roll slides every series forward by k = len(samples[i]) new samples, y <- y[k:] ++ samples[i] for the i-th series in Add
// order: on the device store in place (the store is not sent to the device again) and in each Series' values, which a later
// store rebuild uploads.  Every row holds the same k, 0 <= k <= Length(); the checks come before any device call.  A sharded
// group (SetShard) rolls its own block of series; nothing is exchanged.  When the device fails part-way the store is dropped
// and rebuilt from the unchanged values by the next call that needs it, so a failed Roll has no effect.
func (g *Group) Roll(samples [][]float64) error {
	if len(samples) != len(g.series) {
		return fmt.Errorf("Roll: %d rows of samples for %d series", len(samples), len(g.series))
	}
	if len(samples) == 0 {
		return nil
	}
	k := len(samples[0])
	for i, r := range samples {
		if len(r) != k {
			return fmt.Errorf("Roll: row %d has %d samples, row 0 has %d", i, len(r), k)
		}
	}
	if k > g.n {
		return fmt.Errorf("Roll: %d new samples exceed the series length %d", k, g.n)
	}
	if k == 0 {
		return nil
	}
	if err := g.syncDevice(); err != nil {
		return err
	}
	per := rollChunkBytes / (8 * k)
	if per < 1 {
		per = 1
	}
	if per > len(samples) {
		per = len(samples)
	}
	buf := make([]float64, 0, per*k)
	for first := 0; first < len(samples); first += per {
		end := first + per
		if end > len(samples) {
			end = len(samples)
		}
		buf = buf[:0]
		for _, r := range samples[first:end] {
			buf = append(buf, r...)
		}
		if rc := C.muse_group_roll(g.store, C.int64_t(first), C.int64_t(end-first), (*C.double)(unsafe.Pointer(&buf[0])), C.int64_t(k)); rc != C.MUSE_OK {
			err := lastError(rc)
			C.muse_group_destroy(g.store)
			g.store = nil
			return err
		}
	}
	for i, s := range g.series {
		v := make([]float64, 0, g.n)
		v = append(v, s.vals[k:]...)
		s.vals = append(v, samples[i]...)
	}
	return nil
}

// keyCols maps label names to device columns; unknown names mean "no series has it", which
// puts every series in one group (labels.go:61-65 skips absent keys).
func (g *Group) keyCols(groupByLabels []string) []int32 {
	if len(groupByLabels) == 0 {
		return nil
	}
	seen := map[string]bool{}
	var cols []int32
	names := append([]string(nil), groupByLabels...)
	sort.Strings(names)
	for _, name := range names {
		if seen[name] {
			continue
		}
		seen[name] = true
		for c, k := range g.cols {
			if k == name {
				cols = append(cols, int32(c))
			}
		}
	}
	if len(cols) == 0 {
		cols = []int32{int32(len(g.cols))}
	}
	return cols
}

// whereCols maps the label set of FilterByLabelValues to device columns and value ids; ok == false when no series can match
// (a key or a value the dictionary does not know).
func (g *Group) whereCols(labels *Labels) (cols, ids []int32, ok bool) {
	for _, k := range labels.Keys() {
		v, _ := labels.Get(k)
		c := sort.SearchStrings(g.cols, k)
		if c == len(g.cols) || g.cols[c] != k {
			return nil, nil, false
		}
		id, seen := g.dict[k][v]
		if !seen {
			return nil, nil, false
		}
		cols = append(cols, int32(c))
		ids = append(ids, id)
	}
	return cols, ids, len(cols) > 0
}

var errNoSeries = errors.New("comparison group is empty")
